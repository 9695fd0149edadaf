#!/usr/bin/env python
"""bench.py — benchmark of the GP-posterior + acquisition hot path (contract: see the prompt / DESIGN.md §6).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--config headline|c2|c3|c4|c5] [--scaling weak|strong]
                    [--dump-outputs DIR]

headline (default, the driver's run)
  metric  : acquisition candidate-points/sec, ExpectedImprovement on an exact GPR with N=4096 training points, fp64
            (BASELINE.json `metric`); workload = the synthetic "headline" config of SURVEY.md §8d (Ackley-10D data, Matern52,
            build_gpr defaults, candidates ~ U[0,1]^10).
  step    : one pass of predict + EI + first-max argmax over the rank's shard of the candidates, then the path's single
            collective — `trieste_b200.parallel.sharded_argmax_local` (one NCCL all-gather of (value, global index, x)).
            weak scaling: every rank owns M candidates; strong scaling: 4e6 candidates in total (SURVEY.md §8d) split N ways.
  value   : whole-job candidates/s with the candidates already resident in HBM.
  e2e     : the same call with HOST buffers (pinned; the pageable figure is reported beside it): H2D of the candidates and
            D2H of all M acquisition values + the best pair are inside the timed region.
  roofline: dominant kernel = the int8 digit GEMM (A = Linv·K* as P exact int8 digit products on tcgen05, P = 15 or 21 as the
            engine picked): achieved = P·N² int8 ops per candidate x candidates per launch / average launch duration from CUDA
            events recorded on the library's stream around every launch of the timed region; peak = 2 x the measured cuBLAS
            bf16 rate of MEASURED_PEAKS.json (int8 dense = 2 x bf16 dense on B200), sustained figure.
c2..c5  : the other BASELINE.json configs through the same package API (one JSON line each; kept under profiles/).
--impl reference : the CPU restatement of the reference's path (oracle/gp_oracle.py; TensorFlow/GPflow are not installable
            here, so there is no baseline/_ref) on all host cores: multi-threaded dtrsm + thread-pool Matern evaluation.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

N_TRAIN = 4096
DIM = 10
M_PER_GPU = 1_193_472  # 21 chunks of 56,832 candidates (= 592 tiles of 96: whole waves for both kernels of a chunk)
M_STRONG_TOTAL = 4_000_000  # SURVEY.md §8d headline batch
METRIC = "acquisition candidate-points/sec (EI on GPR N=4096 fp64)"
UNIT = "candidates/s"


def synth_problem():
    """SURVEY.md §8d headline config: X ~ U[0,1]^10 seed 0, y = Ackley-10, Matern52, lengthscale
    0.2*sqrt(D), variance Var(y), mean mean(y), noise Var(y)/100."""
    from trieste_b200.objectives import ackley

    rng = np.random.default_rng(0)
    X = rng.uniform(size=(N_TRAIN, DIM))
    y = ackley(X)
    return X, y


def clocks_sampler(stop_evt, out):
    """Sample nvidia-smi clocks + throttle reasons during the timed region."""
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    dev = os.environ.get("LOCAL_RANK", "0")
    try:
        p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", dev],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return
    out["proc"] = p
    lines = []

    def reader():
        for ln in p.stdout:
            lines.append(ln.strip())

    t = threading.Thread(target=reader, daemon=True)
    t.start()
    stop_evt.wait()
    p.terminate()
    try:
        p.wait(timeout=5)
    except Exception:
        p.kill()
    t.join(timeout=2)
    out["lines"] = lines


def summarise_clocks(lines):
    sm, mx, pw, reasons = [], [], [], set()
    for ln in lines or []:
        f = [x.strip() for x in ln.split(",")]
        if len(f) < 7:
            continue
        try:
            sm.append(float(f[0]))
            mx.append(float(f[1]))
            pw.append(float(f[2]))
        except ValueError:
            continue
        for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
            if v.lower().startswith("active"):
                reasons.add(name)
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)) if pw else None,
            "reasons": sorted(reasons), "samples": len(sm)}


def dgemm_peak_tflops():
    """Measured fp64 GEMM peak on this GPU (cuBLAS via torch.matmul, 6144^3, best of 5) — context for the fp64-equivalent rate."""
    import torch

    n = 6144
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2.0 * n**3 / (best * 1e-3) / 1e12


# ======================================================================================================================
# CPU arm: the oracle (restatement of the reference path) on the host cores
# ======================================================================================================================
_ORACLE_MODEL = None


def _oracle_model():
    """Oracle model of the headline config, built once (outside every timed region)."""
    global _ORACLE_MODEL
    if _ORACLE_MODEL is None:
        from oracle import gp_oracle as o  # cpu_baseline / reference leg: the checker timed beside the product

        X, y = synth_problem()
        var = float(np.var(y))
        om = o.build_model("matern52", X, y, var, np.full(DIM, 0.2 * math.sqrt(DIM)), var / 100.0, float(np.mean(y)))
        _ORACLE_MODEL = (o, om, o.ei_eta(om))
    return _ORACLE_MODEL


def _blas_info():
    try:
        from threadpoolctl import threadpool_info

        infos = [i for i in threadpool_info() if i.get("user_api") == "blas"]
        return ", ".join(sorted({f"{i.get('internal_api')} {i.get('version')} ({i.get('threading_layer')}, {i.get('architecture')})" for i in infos}))
    except Exception:
        return "unknown"


def cpu_reference_pass(n_chunks, chunk=8192, seed=1):
    """One bounded pass of the CPU restatement (predict + EI + argmax, oracle/gp_oracle.py) over n_chunks x chunk candidates of
    the headline workload on ALL host cores: the two triangular solves run on the BLAS pool with every core (dtrsm), and the
    Matern kernel matrix — which NumPy would evaluate on ONE core — is evaluated in column slabs on a thread pool of the same
    size (oracle.KERNEL_WORKERS; the elementwise loops release the GIL).  Returns (candidates, seconds, best)."""
    o, om, eta = _oracle_model()
    cores = os.cpu_count() or 1
    try:  # torchrun exports OMP_NUM_THREADS=1: give the BLAS pool every host core back
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=cores)
    except Exception:
        pass
    o.KERNEL_WORKERS = cores
    rng = np.random.default_rng(seed)
    Xc = rng.uniform(size=(n_chunks * chunk, DIM))
    t0 = time.perf_counter()
    ei = o.expected_improvement_at(om, Xc, eta, chunk=chunk)
    j = int(np.argmax(ei))
    dt = time.perf_counter() - t0
    o.KERNEL_WORKERS = 1
    return n_chunks * chunk, dt, (float(ei[j, 0]), j)


def cpu_reference_rate(sample_target_s=12.0, reps=5):
    """CPU baseline for the native arm's JSON line: `reps` repetitions of a pass sized for ~sample_target_s / reps seconds,
    median rate.  Returns (candidates/s, description dict)."""
    cores = os.cpu_count() or 1
    n0 = 1
    cpu_reference_pass(n0)  # warm-up (page-in, thread pools)
    n, dt, _ = cpu_reference_pass(n0)
    per_rep = sample_target_s / reps
    n_chunks = int(max(1, min(64, round(n0 * per_rep / max(dt, 1e-3)))))
    rates, total, secs = [], 0, 0.0
    for r in range(reps):
        n, dt, _ = cpu_reference_pass(n_chunks, seed=2 + r)
        rates.append(n / dt)
        total += n
        secs += dt
    return float(np.median(rates)), {"cores": cores, "repetitions": reps, "rates": rates, "candidates": total, "seconds": secs,
                                     "blas": _blas_info()}


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU implementation of the path is TensorFlow/GPflow, which cannot be installed here
    (no wheels, no network) -> the oracle port is timed instead, on rank 0 only, every step a bounded sample."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    _oracle_model()
    n0 = 1
    cpu_reference_pass(n0)
    n, dt, _ = cpu_reference_pass(n0)
    n_chunks = int(max(1, min(64, round(n0 * 4.0 / max(dt, 1e-3)))))  # ~4 s per step
    per_step, total = [], 0
    for i in range(args.warmup + args.steps):
        n, dt, _ = cpu_reference_pass(n_chunks if i >= args.warmup else n0, seed=1 + i)
        if i >= args.warmup:
            per_step.append(dt)
            total += n
    value = total / sum(per_step)
    rates = [n_chunks * 8192 / t for t in per_step]
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * float(np.mean(per_step)), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"headline: EI on GPR N={N_TRAIN} D={DIM} Matern52 fp64, Ackley-10 synthetic (SURVEY.md §8d)",
                   "candidates_per_step": total // max(1, args.steps)},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "blas": _blas_info(),
                         "median_rate": float(np.median(rates)), "repetitions": len(rates),
                         "sample": f"{total} candidates over {args.steps} steps (NumPy/SciPy oracle in chunks of 8192: dtrsm on {cores} BLAS "
                                   f"threads, Matern kernel matrix in {cores} column slabs on a thread pool; TensorFlow/GPflow not "
                                   "installable -> CPU restatement)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ======================================================================================================================
# native arm
# ======================================================================================================================
class Timer:
    """Barrier + synchronize on both sides, CUDA events on the library's stream, max over ranks."""

    def __init__(self, lib, stream, world, warmup):
        self.lib, self.stream, self.world, self.warmup = lib, stream, world, warmup

    def __call__(self, step_fn, steps, profile_handle=None):
        import torch
        import torch.distributed as dist

        for _ in range(self.warmup):
            step_fn()
        if profile_handle is not None:
            self.lib.tb_gp_profile(profile_handle, 1)
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = self.lib.tb_launch_count()
        e0.record(self.stream)
        res = None
        for _ in range(steps):
            res = step_fn()
        e1.record(self.stream)
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        launches = self.lib.tb_launch_count() - l0
        if self.world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms, launches, res


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# 16 MB of float64 values + 16 MB of row numbers; a dump holds at most one array this long, so it stays below 64 MB
DUMP_MAX_ROWS = 2_000_000


def dump_outputs(out_dir, arrays):
    """Write each array of ``arrays`` (name -> array or scalar) as ``out_dir/<name>.npy`` in float64; indices are exact
    below 2**53.  An array of more than DUMP_MAX_ROWS rows is cut to a fixed, seeded sample of its rows, whose row numbers
    are written beside it as ``<name>_rows.npy``, so two builds run with the same arguments dump the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.ndim and a.shape[0] > DUMP_MAX_ROWS:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_MAX_ROWS, replace=False))
            a = a[rows]
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}.npy"), np.atleast_1d(a))


def run_headline(args, rank, world, local_rank):
    import torch

    import trieste_b200 as tb
    from trieste_b200 import _lib
    from trieste_b200.acquisition import ExpectedImprovement
    from trieste_b200.parallel import shard_bounds, sharded_argmax_local

    # ---- model (replicated on every rank; once-per-step precompute is outside the timed region) ----
    X, y = synth_problem()
    ds = tb.Dataset(X, y)
    spec = tb.build_gpr(ds, tb.Box([0.0] * DIM, [1.0] * DIM))
    model = tb.GaussianProcessRegression(spec, device=local_rank)
    model.set_engine(args.engine)
    fn = ExpectedImprovement().prepare_acquisition_function(model, ds)
    products, err_est = model.engine_info()
    lib = _lib.lib()
    h = model.handle

    if args.scaling == "strong":
        total = args.candidates or M_STRONG_TOTAL
        lo, hi = shard_bounds(total, rank, world)
        M, offset = hi - lo, lo
    else:
        M = args.candidates or M_PER_GPU
        total, offset = M * world, rank * M
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1 + rank)
    xc_dev = torch.rand(M, DIM, dtype=torch.float64, device="cuda", generator=gen)  # Box.sample semantics
    xc_pinned = torch.empty(M, DIM, dtype=torch.float64).pin_memory()
    xc_pinned.copy_(xc_dev.cpu())
    xc_pageable = xc_pinned.numpy().copy()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    sp = C.c_void_p()
    _lib.check(lib.tb_gp_stream(h, C.byref(sp)))
    stream = torch.cuda.ExternalStream(sp.value)
    timer = Timer(lib, stream, world, args.warmup)

    def step_device():
        flush.zero_()
        return sharded_argmax_local(fn, xc_dev, offset)

    def make_host_step(xh):
        vals = np.empty((M, 1)) if isinstance(xh, np.ndarray) else None

        def step():
            flush.zero_()
            # the user-facing call with host buffers: values of all M candidates come back to the host as well
            v = fn(xh[:, None, :])
            j = int(np.argmax(np.asarray(v)[:, 0]))
            from trieste_b200.parallel import allgather_best

            return allgather_best(float(np.asarray(v)[j, 0]), offset + j, np.asarray(xh[j]))

        return step

    def step_host_fused(xh):
        best_v, best_i = C.c_double(), C.c_int64()
        vals_host = torch.empty(M, dtype=torch.float64).pin_memory() if not isinstance(xh, np.ndarray) else np.empty(M)
        vp = vals_host.data_ptr() if hasattr(vals_host, "data_ptr") else vals_host.ctypes.data
        xp = xh.data_ptr() if hasattr(xh, "data_ptr") else xh.ctypes.data

        def step():
            from trieste_b200.parallel import allgather_best

            flush.zero_()
            _lib.check(lib.tb_acq_argmax(h, _lib.ACQ_EI, fn.eta, xp, M, vp, C.byref(best_v), C.byref(best_i)))
            j = best_i.value
            pt = xh[j].numpy() if hasattr(xh, "numpy") else xh[j]
            return allgather_best(best_v.value, offset + j, pt)

        step.values = vals_host  # the M acquisition values the last step wrote to the host
        return step

    # ---- clocks during the timed region ----
    stop_evt, clk = threading.Event(), {}
    th = threading.Thread(target=clocks_sampler, args=(stop_evt, clk), daemon=True)
    if rank == 0:
        th.start()
        time.sleep(0.3)

    ms_dev, launches, res = timer(step_device, args.steps, profile_handle=h)
    tg_ms, tg_n, tg_fl = C.c_double(), C.c_int64(), C.c_double()
    lib.tb_gp_profile_read(h, C.byref(tg_ms), C.byref(tg_n), C.byref(tg_fl))
    lib.tb_gp_profile(h, 0)
    step_pinned = step_host_fused(xc_pinned)
    ms_e2e, _, _ = timer(step_pinned, args.steps)
    ms_e2e_pageable, _, _ = timer(step_host_fused(xc_pageable), max(1, min(args.steps, 3)))
    n_pageable = max(1, min(args.steps, 3))

    if rank == 0:
        stop_evt.set()
        th.join(timeout=10)
    clocks = summarise_clocks(clk.get("lines"))
    if args.dump_outputs and rank == 0:
        # device-resident path: what sharded_argmax_local returns; pinned host path: the values tb_acq_argmax wrote
        dump_outputs(args.dump_outputs, {"best_point": res[0], "best_value": res[1], "best_index": res[2],
                                         "ei_values": step_pinned.values.numpy()})

    value = total * args.steps / (ms_dev * 1e-3)
    e2e_value = total * args.steps / (ms_e2e * 1e-3)
    e2e_pageable = total * n_pageable / (ms_e2e_pageable * 1e-3)
    if rank != 0:
        return

    dgemm_tf = dgemm_peak_tflops()
    peaks = load_peaks()
    fp64_eq_tf = tg_fl.value / (tg_ms.value * 1e-3) / 1e12 if tg_ms.value > 0 else 0.0
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    nb = N_TRAIN // 128
    cand_per_launch = tg_fl.value / max(tg_n.value, 1) / (N_TRAIN**2)
    avg_launch_s = tg_ms.value * 1e-3 / max(tg_n.value, 1)
    if products > 0:
        # P exact int8 digit products per fp64 product (DESIGN.md §4b/4c): algorithmic int8 ops = P N^2 per candidate
        # (N^2/2 triangular multiply-adds x 2 ops x P).  int8 dense rate = 2 x the bf16 dense rate on this part
        # (4.5 vs 2.25 POP/s nominal): peak = 2 x the measured cuBLAS bf16 figure (sustained: timed inside a long step)
        ops_per_cand = float(products) * N_TRAIN**2
        achieved = ops_per_cand * cand_per_launch / avg_launch_s / 1e12 if avg_launch_s > 0 else 0.0
        bf16 = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
        peak, roof_unit = 2.0 * bf16, "TOP/s"
        digits = {15: 5, 21: 6, 6: 3, 10: 4}.get(products, 0)
        kernel_name = ("oz5::trigemm_kernel<5> (tcgen05 kind::i8, single pass, 5 TMEM accumulator levels of 96 columns)" if products == 15
                       else "oz::trigemm_i8_kernel (tcgen05 kind::i8, two passes)")
        peak_src = ("of measured: 2 x bf16_tflops_sustained of MEASURED_PEAKS.json (int8 dense = 2 x bf16 dense on B200; the file "
                    "carries no int8 figure); tools/i8_shape_bench.cu measured the MMA issue ceilings: 4596 TOP/s at N=128, "
                    "3943 TOP/s at the N=96 tile this kernel uses (shared-memory operand reads)")
        # HBM: K* digit tiles (digits B / element) written once by the generation kernel and read ~once by the GEMM (L2-friendly order)
        bytes_per_cand = 2.0 * digits * N_TRAIN
        traffic_key = "trigemm5_dram_bytes_per_launch" if products == 15 else "trigemm_i8_dram_bytes_per_launch"
        engine_txt = (f"int8: fp64 operands split error-free into {digits} balanced base-256 int8 digits (tight per-row scales, centred K*), "
                      f"{products} exact digit GEMMs on tcgen05 kind::i8 with int32 TMEM accumulators, fp64 recombination; picked by the "
                      f"a-priori error estimate {err_est:.2e} sigma_f^2 (bar 1e-9); parity to the fp64 oracle at 1e-9 sigma_f^2")
    else:
        achieved, peak, roof_unit = fp64_eq_tf, dgemm_tf, "TFLOP/s"
        kernel_name = "trigemm_kernel<false, EPI_SUMSQ> (fp64 DMMA)"
        peak_src = "of measured: cuBLAS DGEMM 6144^3 in this process (MEASURED_PEAKS.json has no fp64 figure)"
        bytes_per_cand = 8.0 * N_TRAIN * (nb + 1) / 2.0
        traffic_key = "trigemm_dram_bytes_per_launch"
        engine_txt = "fp64: native DMMA triangular GEMM"
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get(traffic_key)
    except Exception:
        pass
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        rate, info = cpu_reference_rate()
        cpu = {"value": rate, "unit": UNIT, "cores": info["cores"], "kind": "port", "blas": info["blas"],
               "repetitions": info["repetitions"], "rates": info["rates"],
               "sample": f"{info['candidates']} candidates of the same workload in {info['seconds']:.1f} s: median of {info['repetitions']} "
                         f"repetitions (NumPy/SciPy oracle in chunks of 8192: dtrsm on {info['cores']} BLAS threads, Matern in "
                         f"{info['cores']} column slabs on a thread pool)"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {
            "engine": engine_txt, "digit_products": products,
            "workload": f"headline: EI on GPR N={N_TRAIN} D={DIM} Matern52 fp64, Ackley-10 synthetic (SURVEY.md §8d)",
            "candidates_per_gpu_per_step": M, "candidates_total_per_step": total,
            "parallelism": f"candidate-sharded x{world} through trieste_b200.parallel.sharded_argmax_local, 1 NCCL all-gather/step",
            "l2": "256 MiB L2 flush between timed iterations; per-chunk K* digit scratch (0.9 GB) also exceeds L2",
        },
        "roofline": {
            "bound": "tensor", "achieved": achieved, "peak": peak, "unit": roof_unit,
            "frac": achieved / peak if peak > 0 else None, "traffic": traffic,
            "kernel": kernel_name, "launches_timed": tg_n.value,
            "avg_launch_ms": avg_launch_s * 1e3, "candidates_per_launch": cand_per_launch,
            "peak_source": peak_src,
            # transparency: the same achieved figure against the other candidates for an int8 denominator
            "frac_of_nominal_int8_4500": (achieved / 4500.0) if products > 0 else None,
            "frac_of_measured_issue_ceiling": (achieved / (3943.0 if products == 15 else 4596.0)) if products > 0 else None,
            "kernel_share_of_step": (tg_ms.value / ms_dev) if ms_dev > 0 else None,
            "fp64_equivalent_tflops": fp64_eq_tf, "fp64_dgemm_peak_tflops": dgemm_tf,
            "hbm": {"algorithmic_bytes_per_candidate": bytes_per_cand,
                    "achieved_gbs": bytes_per_cand * cand_per_launch / avg_launch_s / 1e9 if avg_launch_s > 0 else None,
                    "peak_gbs": hbm_peak,
                    "frac": (bytes_per_cand * cand_per_launch / avg_launch_s / 1e9) / hbm_peak if avg_launch_s > 0 else None,
                    "note": "tensor-pipe bound (N^2 multiply-adds per candidate); HBM fraction reported as the north-star asks"},
        },
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": total * DIM * 8, "d2h_bytes_per_step": total * 8 + world * 16,
                "ms_per_step": ms_e2e / args.steps, "host_memory": "pinned",
                "pageable": {"value": e2e_pageable, "ms_per_step": ms_e2e_pageable / n_pageable, "steps": n_pageable}},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "best": {"value": res[1], "global_index": res[2]},
    }
    print(json.dumps(line), flush=True)


# ---- the other BASELINE.json configs (profiles/, not the driver's run) ---------------------------------------------------
def _model(tb, obj, N, D, local_rank, dtype=np.float64, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.uniform(size=(N, D)).astype(dtype)
    y = obj(X.astype(np.float64)).astype(dtype)
    space = tb.Box([0.0] * D, [1.0] * D)
    ds = tb.Dataset(X, y)
    return tb.GaussianProcessRegression(tb.build_gpr(ds, space), device=local_rank), ds, space


def run_config(args, rank, world, local_rank):
    import torch

    import trieste_b200 as tb
    from trieste_b200 import _lib
    from trieste_b200.objectives import ackley, hartmann_6
    from trieste_b200.parallel import (shard_bounds, sharded_argmax_local, sharded_multistart_local,
                                       sharded_thompson_argmin_local)

    lib = _lib.lib()
    cfg = args.config
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1 + rank)

    def shard(total_default):
        total = args.candidates or total_default
        if args.scaling == "strong":
            lo, hi = shard_bounds(total, rank, world)
            return hi - lo, lo, total
        m = total // 8 if cfg in ("c4", "c5") else total  # weak: one GPU's share of the 8-way config
        return m, rank * m, m * world

    if cfg == "c2":
        from trieste_b200.acquisition import ExpectedImprovement

        model, ds, space = _model(tb, hartmann_6, 1024, 6, local_rank)
        fn = ExpectedImprovement().prepare_acquisition_function(model, ds)
        M, off, total = shard(1_000_000)
        x = torch.rand(M, 6, dtype=torch.float64, device="cuda", generator=gen)
        step = lambda: sharded_argmax_local(fn, x, off)  # noqa: E731
        units, unit, name = total, "candidates/s", "C2 Hartmann6 GPR N=1024 fp64 EI random search over 1e6 candidates"
        handle = model.handle
    elif cfg == "c3":
        from trieste_b200.acquisition import BatchMonteCarloExpectedImprovement

        model, ds, space = _model(tb, ackley, 4096, 10, local_rank)
        q, S = 8, 512
        fn = BatchMonteCarloExpectedImprovement(S).prepare_acquisition_function(model, ds)
        fn._sampler.set_eps(np.random.default_rng(3).standard_normal((q, S)))
        B, off, total = shard(65_536)
        x = torch.rand(B, q, 10, dtype=torch.float64, device="cuda", generator=gen)

        def step():
            v = fn(x)
            j = int(torch.argmax(v[:, 0])) if hasattr(v, "device") else int(np.argmax(np.asarray(v)[:, 0]))
            from trieste_b200.parallel import allgather_best

            return allgather_best(float(v[j, 0]), off + j, None)

        units, unit, name = total, "q-batches/s", "C3 Ackley-10 GPR N=4096 fp64 BatchMonteCarloExpectedImprovement q=8 S=512"
        handle = model.handle
    elif cfg == "c4":
        from trieste_b200.sampler import RandomFourierFeatureTrajectorySampler

        model, ds, space = _model(tb, hartmann_6, 1024, 6, local_rank)
        nb = args.batch
        sampler = RandomFourierFeatureTrajectorySampler(model, 2048, seed=0)  # same seed on every rank: identical W, b, theta
        traj = sampler.get_trajectory()
        traj._batch_size = nb
        traj.resample()
        traj._initialized = True
        M, off, total = shard(10_000_000)
        x = torch.rand(M, 6, dtype=torch.float64, device="cuda", generator=gen)
        step = lambda: sharded_thompson_argmin_local(traj, x, off)  # noqa: E731
        units, unit = total, "candidates/s"
        name = f"C4 Hartmann6 RFF F=2048, batch Thompson sampling ({nb} trajectories per pass) over 1e7 candidates"
        handle = model.handle
    else:  # c5
        from trieste_b200.acquisition import LogExpectedImprovement

        def rff_obj(xx, terms=64, seed=2):
            r = np.random.default_rng(seed)
            w = r.standard_normal((terms, xx.shape[-1])) * 3.0
            ph = r.uniform(0, 2 * math.pi, terms)
            a = r.standard_normal(terms) / math.sqrt(terms)
            return (np.cos(xx @ w.T + ph) * a).sum(-1, keepdims=True)

        model, ds, space = _model(tb, rff_obj, 8192, 20, local_rank, dtype=np.float32)
        fn = LogExpectedImprovement().prepare_acquisition_function(model, ds)
        R, off, total = shard(100_000)
        x0 = np.random.default_rng(10 + rank).uniform(size=(R, 20))
        lo_b, up_b = np.zeros(20), np.ones(20)

        def optimise(starts):
            ok, f, xs, nfev = fn.maximize_from(starts, lo_b, up_b, maxiter=args.maxiter)
            return xs, f

        step = lambda: sharded_multistart_local(optimise, x0, off)  # noqa: E731
        units, unit = total, "starts/s"
        name = f"C5 Synthetic-20D GPR N=8192 fp32 log-EI, generate_continuous_optimizer multi-starts (L-BFGS maxiter {args.maxiter}) with NCCL argmax"
        handle = model.handle

    sp = C.c_void_p()
    _lib.check(lib.tb_gp_stream(handle, C.byref(sp)))
    stream = torch.cuda.ExternalStream(sp.value)
    timer = Timer(lib, stream, world, args.warmup)
    stop_evt, clk = threading.Event(), {}
    th = threading.Thread(target=clocks_sampler, args=(stop_evt, clk), daemon=True)
    if rank == 0:
        th.start()
        time.sleep(0.3)
    t0 = time.perf_counter()
    ms, launches, res = timer(step, args.steps)
    wall = time.perf_counter() - t0
    if rank == 0:
        stop_evt.set()
        th.join(timeout=10)
        if args.dump_outputs:
            names = ("best_value", "best_index", "best_point") if cfg == "c3" else ("best_point", "best_value", "best_index")
            dump_outputs(args.dump_outputs, {n: a for n, a in zip(names, res) if a is not None})
        # C5 runs host-side bookkeeping between device rounds: its step time is taken from the stream events like the others;
        # the wall clock of the timed loop (incl. warm-up) is reported beside it
        line = {"metric": name, "value": units * args.steps / (ms * 1e-3), "unit": unit, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": "f32" if cfg == "c5" else "f64", "data": "synthetic",
                "config": {"workload": name, "units_total_per_step": units, "digit_products": model.engine_info()[0],
                           "parallelism": f"sharded x{world} through trieste_b200.parallel, 1 NCCL all-gather/step"},
                "gpu_launches": int(launches), "clocks": summarise_clocks(clk.get("lines")), "wall_s_incl_warmup": wall}
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="headline", choices=["headline", "c2", "c3", "c4", "c5"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--candidates", type=int, default=0, help="candidates per GPU per step (weak) / in total (strong); 0 = the config's default")
    ap.add_argument("--batch", type=int, default=8, help="c4: trajectories per Thompson pass")
    ap.add_argument("--maxiter", type=int, default=30, help="c5: L-BFGS iterations per start")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--engine", default="int8", choices=["int8", "int8x21", "fp64"],
                    help="variance GEMM engine: int8 = fp64-accurate digit split on the INT8 tensor cores, product count picked from the "
                         "error estimate (default); int8x21 = the full 21 products; fp64 = native DMMA")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float64; rank 0's "
                         "values for several GPUs); headline: the winner of the device-resident path and the acquisition "
                         "values of the pinned host path")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to --impl native")
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import __graft_entry__ as g

    g.build()
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.config == "headline":
            run_headline(args, rank, world, local_rank)
        else:
            run_config(args, rank, world, local_rank)
    finally:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
