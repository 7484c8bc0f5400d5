#!/usr/bin/env python
"""
bench.py -- EI candidate evaluations per second on B200 (BASELINE.json metric).

Workload (config #2 of BASELINE.json, SURVEY.md 8d): GaussianProcess, SE-ARD kernel, d=6, N=2048
observations (X ~ U[0,1]^6 seed 0, Y = -Hartman6(X), theta = [.53,.57,2.5,.34,.27,.35], noise 0.1,
xi 0.01), EI over 2^20 uniform random candidates per GPU (seed 1 + rank).  A "step" is one pass of the
hot path (K1 cross-covariance -> K2 triangular DMMA GEMM + reduction -> K3 EI epilogue -> argmax) over
the whole candidate set.  Wide batches take the library's default arithmetic: sigma^2 through the INT8 tensor-core emulation of
the FP64 triangular GEMM (tcgen05.mma kind::i8, exact integer digit products, error of the FP64 GEMM); `--fp64` makes the FP64
DMMA kernels the main arm, and whichever is not the main arm is timed beside it.  With N>1 every rank scores its own
2^20-candidate shard (weak scaling) and the ranks all-reduce the (EI, global index) argmax over NCCL each step; a second,
strong-scaling leg splits rank 0's candidate set over the ranks and checks the NCCL argmax against the single-GPU one.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference      # the reference's own C++ evaluator on the host cores
    python bench.py --dump-outputs DIR    # also write what the last timed step computed, DIR/<name>.npy

torch is used only for the multi-process rendezvous (gloo) -- never for device work.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time
from ctypes import POINTER, c_double, c_float, c_int, c_long

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

THETA = [.53, .57, 2.5, .34, .27, .35]          # ego/utils/testfunctions.py:287
NOISE, XI = 0.1, 0.01
METRIC, UNIT = "EI candidate evals/sec (N=2048, d=6)", "evals/s"

_H6_A = np.array([[10, 3, 17, 3.5, 1.7, 8], [.05, 10, 17, .1, 8, 14], [3, 3.5, 1.7, 10, 17, 8], [17, 8, .05, 10, .1, 14]])
_H6_C = np.array([1, 1.2, 3, 3.2])
_H6_P = np.array([[.1312, .1696, .5569, .0124, .8283, .5886], [.2329, .4135, .8307, .3736, .1004, .9991],
                  [.2348, .1451, .3522, .2883, .3047, .6650], [.4047, .8828, .8732, .5743, .1091, .0381]])


def hartman6_neg(X):
    e = np.sum(_H6_A[None, :, :] * (X[:, None, :] - _H6_P[None, :, :]) ** 2, axis=2)
    return np.sum(_H6_C[None, :] * np.exp(-e), axis=1)


def synthetic_model(n_obs, d=6):
    rs = np.random.RandomState(0)
    X = rs.rand(n_obs, d)
    return X, hartman6_neg(X)


def synthetic_candidates(M, d, rank):
    return np.ascontiguousarray(np.random.RandomState(1 + rank).rand(M, d))


def sobol_block(d, start, n):
    """rows [start, start+n) of the unscrambled Sobol sequence in d dimensions (config #4's candidate set)"""
    import warnings
    from scipy.stats import qmc
    eng = qmc.Sobol(d=d, scramble=False)
    if start:
        eng.fast_forward(start)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")          # "n is not a power of 2": shards and CPU samples are index ranges on purpose
        return np.ascontiguousarray(eng.random(n))


class Workload(object):
    """the two bench lines: BASELINE.json configs[1] (default, weak scaling) and configs[3] (strong scaling)"""

    def __init__(self, args, world):
        self.id = args.workload
        if self.id == 4:
            self.N, self.d = 8192, 10
            self.total = args.candidates if args.candidates else 1 << 24
            self.M = self.total // world                   # strong scaling: the 16M Sobol points are sharded by index range
            self.scaling = "strong"
            self.theta = [0.5 + 0.05 * j for j in range(10)]
            self.metric = "EI candidate evals/sec (N=8192, d=10, Matern-5/2 ARD, %d Sobol candidates sharded over the GPUs)" % self.total
        else:
            self.N, self.d = args.n_obs, args.dim
            self.M = args.candidates if args.candidates else 1 << 20
            self.total = self.M * world
            self.scaling = "weak"
            self.theta = THETA[:self.d]
            self.metric = METRIC

    def model_data(self):
        if self.id == 4:
            rs = np.random.RandomState(4)
            X = rs.rand(self.N, self.d)
            return X, np.sin(2 * X).sum(axis=1)
        return synthetic_model(self.N, self.d)

    def kernel(self):
        from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard, MaternKernel5_ard
        return MaternKernel5_ard(self.theta + [1.0]) if self.id == 4 else GaussianKernel_ard(self.theta)

    def candidates(self, rank):
        if self.id == 4:
            return sobol_block(self.d, rank * self.M, self.M)
        return synthetic_candidates(self.M, self.d, rank)

    def config(self):
        if self.id == 4:
            return {"workload": "config #4: GaussianProcess Matern-5/2 ARD d=10, N=8192 observations, EI xi=0.01 over %d unscrambled Sobol "
                                "candidates sharded by index range (%d per GPU), NCCL argmax" % (self.total, self.M),
                    "n_obs": self.N, "dim": self.d, "candidates_per_gpu": self.M, "arithmetic": "libm-erf / floor 1e-8 (libego) mode",
                    "l2": "inputs larger than L2: each step streams the K* slab (N x M x 7 B of INT8 digits = %.1f GB per GPU; 8 B per "
                          "element on the FP64 arm) besides W and the candidates" % (self.N * self.M * 7 / 1e9)}
        return {"workload": "config #2: GaussianProcess SE-ARD d=%d, N=%d observations (Hartman6), EI xi=%.2f over %d uniform random "
                            "candidates per GPU" % (self.d, self.N, XI, self.M),
                "n_obs": self.N, "dim": self.d, "candidates_per_gpu": self.M, "arithmetic": "libm-erf / floor 1e-8 (libego) mode",
                "l2": "inputs larger than L2: each step streams the K* slab (N x M x 7 B of INT8 digits = %.1f GB; 8 B per element on the "
                      "FP64 arm) besides W and the candidates" % (self.N * self.M * 7 / 1e9)}


def kernel_sass_sha16(kernel):
    """sha256 (first 16 hex digits) of the SASS instruction text of every instantiation of `kernel` in the shipped library"""
    import hashlib
    import re
    from ibo_b200 import _lib
    txt = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=120).stdout
    h, on = hashlib.sha256(), False
    for ln in txt.splitlines():
        if "Function :" in ln:
            on = kernel in ln
        elif on:
            m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", ln)
            if m:
                h.update(m.group(1).strip().encode())
    return h.hexdigest()[:16]


def fp64_peak_crosscheck(clocks):
    """two independent figures beside the live DMMA peak: the datasheet arithmetic at the clock sampled during the run, and the
    cuBLAS DGEMM rate measured on this pool in round 1 (profiles/r01_cublas_dgemm.json)"""
    out = {}
    try:
        mhz = clocks.get("sm_mhz") or 1965.0
        out["datasheet_tflops"] = 148 * 64 * 2 * mhz * 1e6 / 1e12          # 64 FP64 FMA per SM per clock
        out["datasheet_at_mhz"] = mhz
    except Exception:
        pass
    try:
        out["cublas_dgemm_tflops_round1"] = json.load(open(os.path.join(ROOT, "profiles", "r01_cublas_dgemm.json")))["cublas_dgemm_tflops"]
    except Exception:
        pass
    return out


DUMP_MAX_SCORES = 1 << 21      # 16 MB of scores and 16 MB of their indices: a dump stays below 64 MB at any candidate count


def dump_outputs(dirname, arrays):
    """--dump-outputs: every array as DIR/<name>.npy in float64"""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.asarray(a, dtype=np.float64))


def score_sample(scores):
    """all the scores of a step, or a fixed seeded sample of DUMP_MAX_SCORES of them beside their candidate indices"""
    if len(scores) <= DUMP_MAX_SCORES:
        return {"ei": scores}
    idx = np.sort(np.random.RandomState(0).choice(len(scores), DUMP_MAX_SCORES, replace=False))
    return {"ei": scores[idx], "ei_index": idx}


def flops_per_candidate_k2(N):
    """algorithmic FP64 flops of the dominant kernel per candidate: TRSM N^2 + the two fused N-long
    reductions 4N (SURVEY.md 8d: F(N,d) = N^2 + N(2d+8); the remaining N(2d+4) belong to K1)."""
    return float(N) * N + 4.0 * N


# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, rank=0, world=1):
        """one sampler per node: rank 0 watches every GPU of the job (eight polling nvidia-smi processes would themselves disturb
        the latency-bound workloads); the other ranks report nothing"""
        self.idx = ",".join(str(i) for i in range(world)) if world > 1 else str(gpu_index)
        self.proc, self.lines, self.active = None, [], rank == 0

    def start(self):
        if not self.active:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.idx, "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.active:
            return None
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": float(min(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "gpus": self.idx, "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own C++ evaluator (oracle/_ref, built from the untouched sources) or,
# if that did not travel, the plain-C oracle port
# ------------------------------------------------------------------------------------------------
def reference_evaluator():
    pd = POINTER(c_double)
    har = os.path.join(ROOT, "oracle", "_ref", "libego_harness.so")
    if os.path.exists(har):
        H = ctypes.CDLL(har)
        H.ref_set_model.argtypes = [c_int, pd, pd, pd, c_int, c_int, pd, c_int, pd, pd, c_double, pd, pd, c_double, c_double]
        H.ref_eval.argtypes = [c_int, c_long, pd, pd, pd, pd, c_int]
        cores = os.cpu_count() or 1

        def run(invR, X, Y, hyper, Xs):
            z = np.zeros(1)
            dp = lambda a: a.ctypes.data_as(pd)
            H.ref_set_model(X.shape[1], dp(invR), dp(X), dp(Y), X.shape[0], 0, dp(hyper), 0, dp(z), dp(z), 0.0, dp(z), dp(z), XI, NOISE)
            out = np.empty(len(Xs))
            t0 = time.perf_counter()
            H.ref_eval(0, len(Xs), dp(Xs), dp(out), None, None, cores)
            return time.perf_counter() - t0, out
        return "reference", cores, run
    port = os.path.join(ROOT, "oracle", "_build", "liboracle_port.so")
    if not os.path.exists(port):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")])
    P = ctypes.CDLL(port)
    P.port_eval.argtypes = [c_int, pd, pd, pd, c_int, c_int, pd, c_int, pd, pd, c_double, pd, pd, c_double, c_double, c_int, c_long, pd, pd, pd, pd]

    def run(invR, X, Y, hyper, Xs):
        z = np.zeros(1)
        dp = lambda a: a.ctypes.data_as(pd)
        out = np.empty(len(Xs))
        t0 = time.perf_counter()
        P.port_eval(X.shape[1], dp(invR), dp(X), dp(Y), X.shape[0], 0, dp(hyper), 0, dp(z), dp(z), 0.0, dp(z), dp(z), XI, NOISE, 0,
                    len(Xs), dp(Xs), dp(out), None, None)
        return time.perf_counter() - t0, out
    return "port", 1, run


def reference_inputs(wl):
    """model arrays in the layout cdirectGP hands to acqmaxGP (ego/acquisition/__init__.py:365-391).
    The reference's C++ has no Matern-5/2 ARD kernel (SURVEY 8a-3), so for config #4 its evaluator is timed with its
    SE-ARD kernel on the same X, Y, theta: its cost -- N kernel values + two dense N x N mat-vecs per candidate
    (cpp/optimizeGP.cpp:57-191) -- does not depend on the kernel."""
    from oracle import ibo_oracle as orc          # allowed here: cpu_baseline / --impl reference legs only
    X, Y = wl.model_data()
    X = np.ascontiguousarray(X); Y = np.ascontiguousarray(Y)
    gp = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, wl.theta, wl.d), X, Y, NOISE)
    return np.ascontiguousarray(gp.invR()), X, Y, np.ascontiguousarray(np.array(wl.theta))


def cpu_baseline(wl, seconds=12.0):
    """SURVEY 8d: (i) the reference's C++ evaluator on all host threads (the headline baseline) and on ONE core; (ii) the reference's
    NumPy path restated scalar-faithfully (two general LU solves against L per candidate, gaussianprocess/__init__.py:209-210) and the
    vectorised triangular-solve variant for context.  Every leg is a bounded sample of the workload's candidates."""
    from oracle import ibo_oracle as orc          # allowed here: cpu_baseline / --impl reference legs only
    kind, cores, run = reference_evaluator()
    invR, X, Y, hyper = reference_inputs(wl)
    gen = (lambda n: sobol_block(wl.d, 0, n)) if wl.id == 4 else (lambda n: synthetic_candidates(n, wl.d, 0))
    probe = gen(4 * cores)
    t, _ = run(invR, X, Y, hyper, probe)
    n = int(min(max(len(probe) * seconds / max(t, 1e-6), 4 * cores), 200000))
    Xs = gen(n)
    t, _ = run(invR, X, Y, hyper, Xs)
    what = "reference cpp/optimizeGP.cpp GP_Maximizer::negei via oracle/_ref" if kind == "reference" else "oracle/oracle_port.c"
    if wl.id == 4:
        what += "; SE-ARD kernel, the reference has no Matern-5/2 ARD"
    out = {"value": n / t, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": "%d of the workload's candidates, %.1f s on %d host threads (%s)" % (n, t, cores, what)}
    try:    # one core (the reference is single-threaded; the harness fans candidates out over threads)
        n1 = max(8, int(n / max(cores, 1) * 3.0 / max(t, 1e-6)))
        n1 = min(n1, 20000)
        if kind == "reference":
            pd = POINTER(c_double)
            H = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libego_harness.so"))
            H.ref_eval.argtypes = [c_int, c_long, pd, pd, pd, pd, c_int]
            X1 = gen(n1); o1 = np.empty(n1)
            t0 = time.perf_counter()
            H.ref_eval(0, n1, X1.ctypes.data_as(pd), o1.ctypes.data_as(pd), None, None, 1)
            t1 = time.perf_counter() - t0
            out["single_core"] = {"value": n1 / t1, "unit": UNIT, "cores": 1, "sample": "%d candidates, %.1f s, same evaluator on one thread" % (n1, t1)}
    except Exception as e:
        out["single_core"] = {"error": str(e)}
    try:    # NumPy path of the reference, scalar-faithful: posterior() per candidate with two general solves against L
        kspec = orc.KernelSpec(orc.K_MATERN5_ARD if wl.id == 4 else orc.K_SE_ARD, list(wl.theta) + ([1.0] if wl.id == 4 else []), wl.d)
        gpo = orc.GPOracle(kspec, X, Y, NOISE)
        ns = 6 if wl.N > 4096 else 16
        Xn = gen(ns)
        t0 = time.perf_counter()
        for x in Xn:
            mu_, s2_ = gpo.posterior_scalar(x)
            orc.ei_py(mu_, s2_, float(np.max(Y)), XI)
        tn = time.perf_counter() - t0
        nv = 2048
        Xv = gen(nv)
        t0 = time.perf_counter()
        mu_, s2_ = gpo.posterior_batch(Xv)
        orc.score(orc.ACQ_EI, "py", mu_, s2_, float(np.max(Y)), XI)
        tv = time.perf_counter() - t0
        out["numpy_path"] = {"value": ns / tn, "unit": UNIT, "cores": os.cpu_count() or 1,
                             "sample": "%d candidates, %.1f s: oracle restatement of GaussianProcess.posterior + EI.negf, two numpy.linalg.solve "
                                       "(general LU) against L per candidate as the reference does (LAPACK threads as configured)" % (ns, tn),
                             "vectorised_triangular_solve": {"value": nv / tv, "unit": UNIT,
                                                             "sample": "%d candidates in one scipy solve_triangular call, %.2f s (not what the reference does)" % (nv, tv)}}
    except Exception as e:
        out["numpy_path"] = {"error": str(e)}
    return out


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    wl = Workload(args, world)
    kind, cores, run = reference_evaluator()
    invR, X, Y, hyper = reference_inputs(wl)
    gen = (lambda n: sobol_block(wl.d, 0, n)) if wl.id == 4 else (lambda n: synthetic_candidates(n, wl.d, 0))
    probe = gen(4 * cores)
    t, _ = run(invR, X, Y, hyper, probe)
    per_step = int(min(max(len(probe) * 4.0 / max(t, 1e-6), 4 * cores), 100000))      # ~4 s of CPU work per step
    Xs = gen(per_step)
    for _ in range(args.warmup):
        run(invR, X, Y, hyper, Xs[: max(4 * cores, per_step // 8)])
    times = [run(invR, X, Y, hyper, Xs)[0] for _ in range(args.steps)]
    tt = float(np.sum(times))
    value = per_step * args.steps / tt
    sample = "each step = %d candidates of the workload on %d host threads" % (per_step, cores)
    line = {"impl": "reference", "metric": wl.metric, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tt / args.steps, "higher_is_better": True, "scaling": wl.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": wl.config(),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# extra measurements: `maximizeEI wall ms` half of the BASELINE metric, model build, other configs
# ------------------------------------------------------------------------------------------------
def ref_acqmax(invR, X, Y, hyper, kind, lb, ub, xi, noise, maxiter, maxsample):
    """the reference's own acqmaxGP (oracle/_ref/libego.so) timed on one host core (it is single-threaded)"""
    pd = POINTER(c_double)
    path = os.path.join(ROOT, "oracle", "_ref", "libego.so")
    if not os.path.exists(path):
        return None
    E = ctypes.CDLL(path)
    E.acqmaxGP.restype = pd
    E.acqmaxGP.argtypes = [c_int, pd, pd, pd, pd, pd, c_int, c_int, c_int, pd, c_int, pd, pd, c_double, pd, pd,
                           c_double, c_double, c_int, c_int, c_int]
    dp = lambda a: a.ctypes.data_as(pd)
    z = np.zeros(1)
    t0 = time.perf_counter()
    res = E.acqmaxGP(X.shape[1], dp(lb), dp(ub), dp(invR), dp(X), dp(Y), X.shape[0], 0, kind, dp(hyper), 0, dp(z), dp(z), 0.0,
                     dp(z), dp(z), xi, noise, maxiter, 10 ** 6, maxsample)
    t = time.perf_counter() - t0
    return {"wall_ms": 1e3 * t, "opt": -res[0], "optx": [res[i + 1] for i in range(X.shape[1])]}


def run_suite(args):
    from ibo_b200 import _lib
    from ibo_b200.acquisition import cdirectGP, maximizeEI
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard, MaternKernel5_ard
    from oracle import ibo_oracle as orc           # reference-side inputs (inv(R)) for the CPU leg only
    _lib.require_gpu()
    out = []

    def emit(d):
        out.append(d)
        print(json.dumps(d), flush=True)

    # warm the context / kernels
    GaussianProcess(GaussianKernel_ard([1.0, 1.0]), np.random.rand(300, 2), np.random.rand(300)).model
    # ---- config #1: demo.py-style maximizeEI, Branin N=50, d=2, 50 DIRECT iterations ----
    bounds = [[-5., 10.], [0., 15.]]
    X = np.array(orc.lhc_sample(bounds, 50, seed=0)); Y = -orc.branin(X) / 100.0
    t0 = time.perf_counter()
    gp = GaussianProcess(GaussianKernel_ard([3.4, 10.0]), X, Y, noise=0.1)
    gp.model
    t_build = time.perf_counter() - t0
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        opt, optx = maximizeEI(gp, bounds, xi=0.01, maxiter=50, maxtime=10 ** 6, maxsample=10000)
        ts.append(time.perf_counter() - t0)
    o = orc.GPOracle(orc.KernelSpec(0, [3.4, 10.0], 2), X, Y, 0.1)
    b = np.array(bounds)
    ref = ref_acqmax(np.ascontiguousarray(o.invR()), np.ascontiguousarray(X), np.ascontiguousarray(Y), np.array([3.4, 10.0]), 0,
                     np.ascontiguousarray(b[:, 0]), np.ascontiguousarray(b[:, 1]), 0.01, 0.1, 50, 10000)
    emit({"suite": "config1_maximizeEI", "N": 50, "d": 2, "maxiter": 50, "wall_ms": 1e3 * min(ts), "model_build_ms": 1e3 * t_build,
          "nsamples": cdirectGP.last["nsamples"], "opt": opt, "optx": list(optx), "reference_acqmaxGP": ref,
          "same_point": bool(ref and np.allclose(optx, ref["optx"], atol=1e-12))})
    # ---- model build (R, Cholesky, W, packing) ----
    for N in (2048, 4096, 8192):
        Xb, Yb = synthetic_model(N, 6)
        best = 1e9
        for _ in range(2):
            t0 = time.perf_counter()
            g = GaussianProcess(GaussianKernel_ard(THETA), Xb, Yb, noise=NOISE)
            g.model
            best = min(best, time.perf_counter() - t0)
            del g
        emit({"suite": "model_build", "N": N, "d": 6, "wall_ms": 1e3 * best, "gflop": 2 * N ** 3 / 3 / 1e9})
    # ---- addData on a resident model: device rank-1 append (ibo_model_append) vs rebuilding the factor ----
    for N in (2048, 8192):
        Xb, Yb = synthetic_model(N + 32, 6)
        g = GaussianProcess(GaussianKernel_ard(THETA), Xb[:N], Yb[:N], noise=NOISE)
        g.model
        g.addData(Xb[N], Yb[N])                      # warm the append kernels
        t0 = time.perf_counter()
        for i in range(N + 1, N + 32):
            g.addData(Xb[i], Yb[i])
        t_app = (time.perf_counter() - t0) / 31
        t0 = time.perf_counter()
        g._invalidate(); g.model
        t_reb = time.perf_counter() - t0
        emit({"suite": "addData_append", "N": N, "d": 6, "append_ms_per_point": 1e3 * t_app, "rebuild_ms": 1e3 * t_reb})
        del g
    # ---- maximizeEI at the headline model size (N=2048, d=6), default budget ----
    Xb, Yb = synthetic_model(2048, 6)
    gp = GaussianProcess(GaussianKernel_ard(THETA), Xb, Yb, noise=NOISE)
    gp.model
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        opt, optx = maximizeEI(gp, [[0., 1.]] * 6, xi=XI, maxiter=50, maxtime=10 ** 6, maxsample=10000)
        ts.append(time.perf_counter() - t0)
    ns = cdirectGP.last["nsamples"]
    o = orc.GPOracle(orc.KernelSpec(0, THETA, 6), Xb, Yb, NOISE)
    ref = ref_acqmax(np.ascontiguousarray(o.invR()), np.ascontiguousarray(Xb), np.ascontiguousarray(Yb), np.array(THETA), 0,
                     np.zeros(6), np.ones(6), XI, NOISE, 50, 400)      # bounded: ~400 samples of the reference (4N^2 flops each)
    emit({"suite": "maximizeEI_N2048", "N": 2048, "d": 6, "maxiter": 50, "maxsample": 10000, "wall_ms": 1e3 * min(ts), "nsamples": ns,
          "ms_per_1000_samples": 1e6 * min(ts) / ns, "opt": opt,
          "reference_acqmaxGP_maxsample400": ref})
    # ---- hyper-parameter learning: one nlml + gradient evaluation (ibo_nlml), SE-ARD + magnitude ----
    for N in (2048, 4096):
        Xb, Yb = synthetic_model(N, 6)
        hy = list(THETA) + [1.0]
        _lib.nlml(_lib.KERNEL_SE_ARD, hy, Xb, Yb, 1e-3)
        tv, tg = [], []
        for _ in range(3):
            t0 = time.perf_counter(); v = _lib.nlml(_lib.KERNEL_SE_ARD, hy, Xb, Yb, 1e-3, want_grad=False)[0]; tv.append(time.perf_counter() - t0)
            t0 = time.perf_counter(); v, gr = _lib.nlml(_lib.KERNEL_SE_ARD, hy, Xb, Yb, 1e-3); tg.append(time.perf_counter() - t0)
        emit({"suite": "nlml", "N": N, "d": 6, "nhyper": 7, "value_ms": 1e3 * min(tv), "value_and_gradient_ms": 1e3 * min(tg),
              "nlml": v, "gflop_value_and_gradient": N ** 3 / 1e9})
    # ---- config #4 slice: Matern-5/2 ARD d=10, N=8192, 2^18 Sobol-like candidates on one GPU ----
    rs = np.random.RandomState(4)
    X4 = rs.rand(8192, 10); Y4 = np.sin(2 * X4).sum(axis=1)
    th4 = [0.5 + 0.05 * j for j in range(10)] + [1.0]
    gp4 = GaussianProcess(MaternKernel5_ard(th4), X4, Y4, noise=0.1)
    m4 = gp4.model
    try:
        from scipy.stats import qmc
        C4 = np.ascontiguousarray(qmc.Sobol(d=10, scramble=False).random_base2(18))
    except Exception:
        C4 = rs.rand(1 << 18, 10)
    rc = _lib.ResidentCandidates(m4, C4)
    rc.score(_lib.ACQ_EI, Y4.max(), 0.01)
    best4, idx4, ms4 = rc.score(_lib.ACQ_EI, Y4.max(), 0.01, _lib.FLAG_PROFILE)
    pr = m4.profile()
    F = 8192.0 ** 2 + 8192 * (2 * 10 + 8)
    emit({"suite": "config4_slice", "N": 8192, "d": 10, "candidates": len(C4), "ms": ms4, "evals_per_s": len(C4) / (ms4 * 1e-3),
          "algorithmic_tflops": len(C4) * F / (ms4 * 1e-3) / 1e12, "k1_ms": pr["k1_ms"], "k2_ms": pr["k2_ms"], "k3_ms": pr["k3_ms"]})
    rc.close()
    del gp4, m4
    # ---- config #3: PrefGaussianProcess (Laplace) d=4, 500 pairwise preferences, fastUCBGallery of 4 ----
    from ibo_b200.acquisition import fastUCBGallery
    from ibo_b200.gaussianprocess import PrefGaussianProcess
    b3 = [[0., 10.]] * 4
    P3 = np.array(orc.lhc_sample(b3, 1000, seed=2))
    prefs = []
    for i in range(500):
        a, b_ = P3[2 * i], P3[2 * i + 1]
        prefs.append((a, b_, 0) if -orc.shekel5(a) > -orc.shekel5(b_) else (b_, a, 0))
    t0 = time.perf_counter()
    pg = PrefGaussianProcess(GaussianKernel_ard([5.146, 4.189, 4.622, 5.843]), prefs, noise=0.1)
    t_fit = time.perf_counter() - t0
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        gal = fastUCBGallery(pg, b3, 4, seed=3)
        ts.append(time.perf_counter() - t0)
    emit({"suite": "config3_pref_gallery", "points": len(pg.X), "prefs": 500, "d": 4, "laplace_fit_host_s": t_fit,
          "fastUCBGallery_wall_ms": 1e3 * min(ts), "gallery": [list(map(float, g)) for g in gal]})
    # ---- config #5: batched-DIRECT maximizeEI d=20, N=4096, 200 iterations ----
    rs = np.random.RandomState(5)
    X5 = rs.rand(4096, 20); Y5 = np.sin(2 * X5).sum(axis=1)
    gp5 = GaussianProcess(GaussianKernel_ard([1.0] * 20), X5, Y5, noise=0.1)
    gp5.model
    t5s = []
    for _ in range(4):      # the first query also builds the model's INT8 digit planes and unit tables
        t0 = time.perf_counter()
        opt5, optx5 = maximizeEI(gp5, [[0., 1.]] * 20, xi=0.01, maxiter=200, maxtime=10 ** 6, maxsample=10 ** 9)
        t5s.append(time.perf_counter() - t0)
    t5 = min(t5s[1:])
    emit({"suite": "config5_direct", "N": 4096, "d": 20, "maxiter": 200, "wall_ms": 1e3 * t5, "first_query_ms": 1e3 * t5s[0], "nsamples": cdirectGP.last["nsamples"],
          "iterations": cdirectGP.last["iterations"], "opt": opt5})
    return out


# ------------------------------------------------------------------------------------------------
def run_direct_workload(args, rank, world, device, dist):
    """BASELINE configs[4]: end-to-end batched-DIRECT maximizeEI, d=20, N=4096, 200 iterations per query.  One process per GPU.
    A query is latency bound (batches of 10^2-10^3 points, ~200 dependent round trips), so the GPUs of a box are used for
    THROUGHPUT: every rank answers its own queries (same model replicated, different incumbents / xi so that the trajectories
    differ), no collective on the data path -- `value` = queries per second over all ranks (weak scaling).  Beside it: the latency
    of ONE query, unsharded on one GPU and with every batch cut into one slice per GPU (IBO_FLAG_SHARD + NCCL all-gather), which
    must give the same point bit for bit."""
    from ibo_b200 import _lib
    from ibo_b200.acquisition import cdirectGP, maximizeEI
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    L = _lib.lib()
    N, d, iters = 4096, 20, 200
    rs = np.random.RandomState(5)
    X = rs.rand(N, d); Y = np.sin(2 * X).sum(axis=1)
    gp = GaussianProcess(GaussianKernel_ard([1.0] * d), X, Y, noise=0.1, device=device)
    gp.model
    bounds = [[0., 1.]] * d

    def sync_all():
        if dist is not None:
            dist.barrier()
        _lib.check(L.ibo_device_synchronize(device))

    def query(shard, xi=0.01):
        return maximizeEI(gp, bounds, xi=xi, maxiter=iters, maxtime=10 ** 6, maxsample=10 ** 9, shard=shard)

    nq = max(args.steps, 1)
    my_xi = [0.01 + 0.003 * ((rank * nq + q) % 7) for q in range(nq)]      # this rank's queries
    for _ in range(max(args.warmup, 1)):
        query(False, my_xi[0])
    sampler = ClockSampler(device, rank, world)
    sync_all()
    sampler.start()
    launches0 = L.ibo_launch_count()
    t0 = time.perf_counter()
    samples = 0
    for q in range(nq):
        last = query(False, my_xi[q])
        samples += cdirectGP.last["nsamples"]
    sync_all()
    t_tp = time.perf_counter() - t0
    launches = L.ibo_launch_count() - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"opt": [last[0]], "optx": last[1]})
    # ---- latency of one query: unsharded on this GPU, and sharded over all GPUs ----
    t0 = time.perf_counter()
    opt1, optx1 = query(False)
    t_single = time.perf_counter() - t0
    n1, its = cdirectGP.last["nsamples"], cdirectGP.last["iterations"]
    t_shard, same = None, None
    if world > 1:
        query(True)
        sync_all()
        t0 = time.perf_counter()
        opt, optx = query(True)
        sync_all()
        t_shard = time.perf_counter() - t0
        same = bool(opt == opt1 and np.array_equal(optx, optx1) and cdirectGP.last["nsamples"] == n1)
    if dist is not None:
        import torch
        t = torch.tensor([t_tp, t_single, t_shard, 0.0 if same else 1.0], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_tp, t_single, t_shard, same = float(t[0]), float(t[1]), float(t[2]), bool(t[3] == 0.0)
        tot = torch.tensor([float(samples)], dtype=torch.float64)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        samples = int(tot[0])
    if rank == 0:
        qps = world * nq / t_tp
        line = {
            "metric": "maximizeEI queries/sec (batched DIRECT, N=4096, d=20, 200 iterations per query)", "value": qps, "unit": "queries/s",
            "n_gpus": world, "steps": nq, "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * t_tp / nq, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "config #5: GaussianProcess SE-ARD d=20, N=4096, maximizeEI through batched DIRECT, 200 iterations per query; "
                                   "every GPU answers its own queries (step = one query per GPU), model replicated, no data-path collective",
                       "n_obs": N, "dim": d, "iterations": its, "nsamples_per_query": n1, "l2": "latency-bound small batches (10^2-10^3 points)"},
            "clocks": clocks, "gpu_launches": int(launches), "evals_per_s": samples / t_tp,
            "single_query": {"unsharded_one_gpu_wall_ms": 1e3 * t_single,
                             "sharded_over_all_gpus_wall_ms": None if t_shard is None else 1e3 * t_shard,
                             "same_result_as_unsharded": same, "opt": opt1,
                             "note": "IBO_FLAG_SHARD cuts every batch of >= 64 x ranks points into one slice per GPU and all-gathers the values over NCCL"},
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": int(n1 * d * 8), "d2h_bytes_per_step": int(n1 * 8),
                    "api": "maximizeEI -> cdirectGP -> ibo_acqmax (host candidates in, values out, every batch)"}}
        print(json.dumps(line))
    if dist is not None:
        L.ibo_comm_destroy()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n-obs", type=int, default=2048)
    ap.add_argument("--dim", type=int, default=6)
    ap.add_argument("--candidates", type=int, default=0, help="per GPU for the default workload (2^20), total for --workload 4 (2^24)")
    ap.add_argument("--workload", type=int, default=2, choices=[2, 4, 5],
                    help="2: BASELINE configs[1] (default, the metric's config); 4: configs[3], N=8192 Matern-5/2 ARD, 16M Sobol, strong scaling; "
                         "5: configs[4], batched-DIRECT maximizeEI d=20, N=4096, 200 iterations, batches sharded over the GPUs (wall ms)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--fp64", action="store_true",
                    help="make the FP64 DMMA kernels (IBO_FLAG_FP64) the main arm instead of the library default (INT8 tensor-core path for wide batches)")
    ap.add_argument("--suite", action="store_true", help="extra measurements (maximizeEI wall ms, model build, configs #1/#4/#5)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed on rank 0 as DIR/<name>.npy (float64): best = [EI, "
                         "global candidate index] of the step's argmax, ei = the EI of every candidate (above %d candidates a fixed "
                         "seeded sample, their indices in ei_index); --workload 5: opt and optx of the last query.  The copy of the "
                         "scores to the host is part of the last timed step; the JSON line says so under dump_outputs" % DUMP_MAX_SCORES)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.suite or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of the timed GPU steps: not with --suite or --impl reference")
    if args.suite:
        return run_suite(args)
    args.warmup = max(args.warmup, 3) if (args.impl == "ours" and args.workload == 2) else max(args.warmup, 1 if args.impl == "ours" else 0)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference_arm(args, rank, world)

    from ibo_b200 import _lib
    from ibo_b200.gaussianprocess import GaussianProcess
    L = _lib.lib()
    ndev = _lib.require_gpu()
    device = local % ndev
    dist = None
    if world > 1:
        import torch.distributed as dist          # rendezvous + host-side max/barrier only (gloo)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo", rank=rank, world_size=world)
        uid = [None]
        if rank == 0:
            buf = ctypes.create_string_buffer(128)
            _lib.check(L.ibo_comm_unique_id(buf))
            uid[0] = buf.raw
        dist.broadcast_object_list(uid, src=0)
        _lib.check(L.ibo_comm_init(device, rank, world, uid[0]))

    if args.workload == 5:
        return run_direct_workload(args, rank, world, device, dist)

    wl = Workload(args, world)
    N, d, M = wl.N, wl.d, wl.M
    X, Y = wl.model_data()
    t0 = time.perf_counter()
    gp = GaussianProcess(wl.kernel(), X, Y, noise=NOISE, device=device)
    model = gp.model                                   # builds R, Cholesky, W = inv(L), packing on the device
    t_factor = time.perf_counter() - t0
    ymax = float(np.max(Y))
    # FP64 tensor-pipe peak first, on a GPU that is not yet power-limited by the INT8 steps (the DMMA path never reaches the cap)
    peak = c_double(0)
    _lib.check(L.ibo_fp64_peak(device, ctypes.byref(peak)))
    Xs = wl.candidates(rank)
    cands = _lib.ResidentCandidates(model, Xs)
    use_i8 = (not args.fp64) and N > 128 and N <= 16384 and d <= 32 and _lib.get_option("int8") == 1
    flags = _lib.FLAG_MODE_CPP | (0 if use_i8 else _lib.FLAG_FP64)
    other_flags = _lib.FLAG_MODE_CPP | (_lib.FLAG_FP64 if use_i8 else _lib.FLAG_INT8)

    def step_resident(scores_out=None):
        best, bidx, ms = cands.score(_lib.ACQ_EI, ymax, XI, flags, scores_out=scores_out)
        gidx = ctypes.c_long(rank * M + bidx)
        sc = c_double(best)
        if world > 1:
            _lib.check(L.ibo_comm_argmax(ctypes.byref(sc), ctypes.byref(gidx)))
        return sc.value, gidx.value

    def sync_all():
        if dist is not None:
            dist.barrier()
        _lib.check(L.ibo_device_synchronize(device))

    for _ in range(args.warmup):
        step_resident()
    # --dump-outputs: the last timed step also copies its scores to the host, into a pinned buffer to keep that copy short
    last_scores = np.empty(M) if (args.dump_outputs and rank == 0) else None
    if last_scores is not None:
        _lib.check(L.ibo_host_register(last_scores.ctypes.data_as(ctypes.c_void_p), last_scores.nbytes))
    sampler = ClockSampler(device, rank, world)
    sync_all()
    sampler.start()
    launches0 = L.ibo_launch_count()
    _lib.check(L.ibo_stream_mark(model.handle, 0))
    tw0 = time.perf_counter()
    for s in range(args.steps):
        best = step_resident(last_scores if s == args.steps - 1 else None)
    _lib.check(L.ibo_stream_mark(model.handle, 1))
    sync_all()
    tw1 = time.perf_counter()
    launches = L.ibo_launch_count() - launches0
    msf = c_float(0)
    _lib.check(L.ibo_stream_elapsed_ms(model.handle, ctypes.byref(msf)))
    clocks = sampler.stop()
    if last_scores is not None:
        _lib.check(L.ibo_host_unregister(last_scores.ctypes.data_as(ctypes.c_void_p)))
        dump_outputs(args.dump_outputs, dict(best=[best[0], best[1]], **score_sample(last_scores)))
    t_dev = msf.value * 1e-3
    t_wall = tw1 - tw0

    # ---- dominant kernel (K2) timing from CUDA events on the launching stream, same workload ----
    def profile_arm(fl, reps):
        k2 = []
        for _ in range(reps):
            cands.score(_lib.ACQ_EI, ymax, XI, fl | _lib.FLAG_PROFILE)
            k2.append(model.profile())
        return min(k2, key=lambda p: p["k2_ms"])
    prof = profile_arm(flags, max(2, min(args.steps, 3)) if wl.id == 2 else 1)
    pk8b, pk8s = c_double(0), c_double(0)
    if N > 128:
        _lib.check(L.ibo_i8_peak2(device, 1.5, ctypes.byref(pk8b), ctypes.byref(pk8s)))
    nbk = (N + 127) // 128
    i8_ops = 2.0 * 28 * 128 * 32 * 4 * (nbk * (nbk + 1) // 2)           # int8 ops per candidate: 28 digit products per 32-deep k-step

    def k2_traffic(kernel, cpl):
        """dram__bytes_read.sum + dram__bytes_write.sum of K2 per launch from the committed ncu --set full capture -- used only when
        the capture was taken from THIS build of the kernel (SASS hash) at this model size"""
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02_k2_traffic.json")))[kernel]
            if tj["n_obs"] != N or tj["sass_sha16"] != kernel_sass_sha16(kernel):
                return None
            return (tj["dram_bytes_read"] + tj["dram_bytes_write"]) * cpl / tj["candidates_per_launch"]
        except Exception:
            return None

    def k2_roofline(p, int8):
        """roofline of the dominant kernel of one arm: algorithmic work per launch / average launch time / live peak"""
        k2_s = p["k2_ms"] * 1e-3 / max(p["k2_launches"], 1)
        cpl = M / max(p["k2_launches"], 1)
        fp64_equiv = cpl * flops_per_candidate_k2(N) / k2_s / 1e12
        if int8:
            ach = cpl * i8_ops / k2_s / 1e12
            return {"bound": "tensor", "achieved": ach, "peak": pk8s.value, "unit": "TOP/s (int8)",
                    "frac": ach / pk8s.value if pk8s.value else None, "traffic": k2_traffic("trigemm_i8_kernel", cpl),
                    "kernel": "trigemm_i8_kernel (K2 on tcgen05.mma kind::i8)", "int8_ops_per_candidate": i8_ops,
                    "candidates_per_launch": cpl, "avg_launch_ms": 1e3 * k2_s,
                    "peak_burst": pk8b.value, "frac_of_burst_peak": ach / pk8b.value if pk8b.value else None,
                    "fp64_equivalent_tflops": fp64_equiv, "fp64_dmma_peak_tflops": peak.value,
                    "peak_source": "ibo_i8_peak2 on this GPU: `peak` = tcgen05.mma kind::i8 from resident pseudo-random operands, back to back for "
                                   "1.5 s, rate over the second half (the kernel runs inside a long, power-capped step: SM clock ~1650 of 1965 MHz); "
                                   "`peak_burst` = best 2 ms launch with near-constant operand bytes at the full clock"}
        return {"bound": "tensor", "achieved": fp64_equiv, "peak": peak.value, "unit": "TFLOP/s", "frac": fp64_equiv / peak.value if peak.value else None,
                "traffic": k2_traffic("trigemm_kernel", cpl), "kernel": "trigemm_kernel (K2 on DMMA.8x8x4)", "flops_per_candidate": flops_per_candidate_k2(N),
                "candidates_per_launch": cpl, "avg_launch_ms": 1e3 * k2_s,
                "peak_source": "live DMMA.8x8x4 issue-rate microbenchmark on this GPU (ibo_fp64_peak); MEASURED_PEAKS.json and the profiling "
                               "guide carry no FP64 figure",
                "peak_crosscheck": fp64_peak_crosscheck(clocks)}

    # ---- the other arithmetic on the same resident candidates (untimed region of the main arm): rate + agreement ----
    other_arm = None
    if wl.id == 2 and N > 128:
        try:
            s_main, s_oth = np.empty(M), np.empty(M)
            b_main = cands.score(_lib.ACQ_EI, ymax, XI, flags, scores_out=s_main)
            b_oth = cands.score(_lib.ACQ_EI, ymax, XI, other_flags, scores_out=s_oth)
            tso = [cands.score(_lib.ACQ_EI, ymax, XI, other_flags)[2] for _ in range(3)]
            po = profile_arm(other_flags, 1)
            other_arm = {"arithmetic": "FP64 DMMA kernels (IBO_FLAG_FP64)" if use_i8 else "INT8 tensor-core path (IBO_FLAG_INT8)",
                         "value": M / (min(tso) * 1e-3), "unit": UNIT, "ms_per_step": min(tso),
                         "kernel_ms_per_step": {"k1_kstar": po["k1_ms"], "k2_trigemm": po["k2_ms"], "k3_epilogue": po["k3_ms"]},
                         "roofline": k2_roofline(po, not use_i8),
                         "max_rel_dEI_between_arms": float(np.max(np.abs(s_main - s_oth) / np.maximum(np.abs(s_oth), 1e-5))),
                         "same_argmax": bool(b_main[1] == b_oth[1])}
        except Exception as e:       # the side leg must never take the main arm down
            other_arm = {"error": str(e)}

    # ---- strong-scaling leg (N > 1): rank 0's candidate set cut into one contiguous slice per rank, NCCL argmax checked ----
    strong = None
    if world > 1 and wl.id == 2:
        from ibo_b200.utils.sharding import shard_range
        X0 = synthetic_candidates(M, d, 0)                       # every rank regenerates rank 0's set (seed 1)
        lo, hi = shard_range(M, world, rank)
        csl = _lib.ResidentCandidates(model, np.ascontiguousarray(X0[lo:hi]))

        def step_strong():
            bs, bi, _ = csl.score(_lib.ACQ_EI, ymax, XI, flags)
            gi = ctypes.c_long(lo + bi); sv = c_double(bs)
            _lib.check(L.ibo_comm_argmax(ctypes.byref(sv), ctypes.byref(gi)))
            return sv.value, gi.value
        for _ in range(2):
            step_strong()
        sync_all()
        nst = max(3, args.steps)
        _lib.check(L.ibo_stream_mark(model.handle, 0))
        for _ in range(nst):
            sbest = step_strong()
        _lib.check(L.ibo_stream_mark(model.handle, 1))
        sync_all()
        ms_s = c_float(0)
        _lib.check(L.ibo_stream_elapsed_ms(model.handle, ctypes.byref(ms_s)))
        single = [0.0, -1.0, 0.0]
        if rank == 0:                                            # the whole set on one GPU: the N = 1 answer and its time
            c0 = _lib.ResidentCandidates(model, X0)
            c0.score(_lib.ACQ_EI, ymax, XI, flags)
            r1 = [c0.score(_lib.ACQ_EI, ymax, XI, flags) for _ in range(2)]
            single = [r1[0][0], float(r1[0][1]), min(r[2] for r in r1)]
            c0.close()
        strong = (ms_s.value / nst, sbest, single)
        csl.close()

    # ---- end to end through the public API with HOST buffers (pinned), copies inside the timed region ----
    int8_arg = None if use_i8 else False
    out = np.empty(M)
    L.ibo_host_register(Xs.ctypes.data_as(ctypes.c_void_p), Xs.nbytes)
    L.ibo_host_register(out.ctypes.data_as(ctypes.c_void_p), out.nbytes)
    for _ in range(2 if wl.id == 2 else 1):
        gp.score_batch(Xs, 'ei', xi=XI, mode='cpp', out=out, int8=int8_arg)
    sync_all()
    te0 = time.perf_counter()
    n_e2e = max(2, min(args.steps, 5)) if wl.id == 2 else max(1, min(args.steps, 2))
    for _ in range(n_e2e):
        sc, b, bi = gp.score_batch(Xs, 'ei', xi=XI, mode='cpp', out=out, int8=int8_arg)
        gidx = ctypes.c_long(rank * M + bi); scv = c_double(b)
        if world > 1:
            _lib.check(L.ibo_comm_argmax(ctypes.byref(scv), ctypes.byref(gidx)))
    sync_all()
    te1 = time.perf_counter()
    t_e2e = (te1 - te0) / n_e2e
    L.ibo_host_unregister(Xs.ctypes.data_as(ctypes.c_void_p))
    L.ibo_host_unregister(out.ctypes.data_as(ctypes.c_void_p))

    # max over ranks
    def rmax(v):
        if dist is None:
            return v
        import torch
        t = torch.tensor([v], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])
    t_dev, t_wall, t_e2e = rmax(t_dev), rmax(t_wall), rmax(t_e2e)
    t_step = max(t_dev, 0.0) / args.steps
    value = world * M / t_step
    # the step's own argmax, checked on every multi-GPU run: every rank must hold the same (score, global index) after
    # ibo_comm_argmax, and it must be the maximum over the ranks' local winners (lowest index on ties)
    argmax_ok = None
    if dist is not None:
        loc = cands.score(_lib.ACQ_EI, ymax, XI, flags)
        allw = [None] * world
        dist.all_gather_object(allw, (loc[0], rank * M + loc[1], best[0], best[1]))
        want = max(((w[0], -w[1]) for w in allw))
        argmax_ok = bool(all((w[2], w[3]) == (want[0], -want[1]) for w in allw))
    F_step = float(N) * N + N * (2.0 * d + 8.0)
    line = {
        "metric": wl.metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_step, "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": wl.config(),
        "clocks": clocks,
        "e2e": {"value": world * M / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(Xs.nbytes), "d2h_bytes_per_step": int(out.nbytes + 16),
                "api": "GaussianProcess.score_batch -> ibo_score_batch (host buffers, pinned)"},
        "gpu_launches": int(launches),
        "roofline": k2_roofline(prof, use_i8),
        "kernel_ms_per_step": {"k1_kstar": prof["k1_ms"], "k2_trigemm": prof["k2_ms"], "k3_epilogue": prof["k3_ms"], "total": prof["total_ms"],
                               "note": "CUDA events around each kernel with the chunks run back to back (IBO_FLAG_PROFILE); the timed steps "
                                       "overlap K1 of chunk c+1 with K2 of chunk c on the INT8 path"},
        "wall_ms_per_step": 1e3 * t_wall / args.steps,
        "model_build_s": t_factor, "best": {"ei": best[0], "index": best[1]},
    }
    # the whole step (K1 + K2 + K3 + argmax) as FP64-equivalent work against the DMMA peak: F(N,d) = N^2 + N(2d+8) flops per candidate
    line["roofline"]["step"] = {"flops_per_candidate": F_step, "fp64_equivalent_tflops": M * F_step / t_step / 1e12,
                                "frac_of_fp64_dmma_peak": (M * F_step / t_step / 1e12 / peak.value) if peak.value else None}
    line["config"]["arithmetic"] += ("; sigma^2 through the INT8 tensor-core emulation of the FP64 GEMM (library default for wide batches), "
                                     "mu as k*.alpha in FP64" if use_i8 else "; FP64 DMMA kernels (IBO_FLAG_FP64)")
    if last_scores is not None:
        line["dump_outputs"] = {"dir": args.dump_outputs, "timed_d2h_bytes": int(last_scores.nbytes),
                                "note": "the last timed step also copied its scores to the host (pinned buffer): that copy is inside "
                                        "the timed region and lowers `value` slightly; runs without --dump-outputs do not copy them"}
    if other_arm is not None:
        line["fp64_dmma_arm" if use_i8 else "int8_arm"] = other_arm
    if argmax_ok is not None:
        line["argmax_is_max_over_ranks"] = argmax_ok
    if strong is not None:
        ms_strong = rmax(strong[0])
        import torch
        sg = torch.tensor(strong[2], dtype=torch.float64)
        dist.broadcast(sg, src=0)
        line["strong"] = {"workload": "rank 0's %d candidates cut into %d contiguous slices (shard_range), NCCL argmax every step" % (M, world),
                          "value": M / (ms_strong * 1e-3), "unit": UNIT, "ms_per_step": ms_strong,
                          "single_gpu_ms_per_step": float(sg[2]), "efficiency_vs_single_gpu": float(sg[2]) / (world * ms_strong),
                          "argmax_matches_single_gpu": bool(strong[1][0] == float(sg[0]) and strong[1][1] == int(sg[1]))}
    # ---- the "maximizeEI wall ms" half of the metric (this rank's GPU; DIRECT is latency bound and is not sharded) ----
    if rank == 0 and wl.id == 2:
        from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
        from ibo_b200.acquisition import cdirectGP, maximizeEI
        from ibo_b200.utils.latinhypercube import lhcSample
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            opt, optx = maximizeEI(gp, [[0., 1.]] * d, xi=XI, maxiter=50, maxtime=10 ** 6, maxsample=10000)
            ts.append(time.perf_counter() - t0)
        mx = {"headline_model": {"N": N, "d": d, "maxiter": 50, "wall_ms": 1e3 * min(ts), "nsamples": cdirectGP.last["nsamples"], "opt": opt}}
        bb = [[-5., 10.], [0., 15.]]                      # config #1: demo.py-style Branin, N = 50, SE-ARD [3.4, 10]
        Xb = np.array(lhcSample(bb, 50, seed=0))
        Yb = -((Xb[:, 1] - (5.1 / (4 * np.pi ** 2)) * Xb[:, 0] ** 2 + 5 * Xb[:, 0] / np.pi - 6) ** 2
               + 10 * (1 - 1 / (8 * np.pi)) * np.cos(Xb[:, 0]) + 10) / 100.0
        gpb = GaussianProcess(GaussianKernel_ard([3.4, 10.0]), Xb, Yb, noise=0.1, device=device)
        gpb.model
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            opt, optx = maximizeEI(gpb, bb, xi=0.01, maxiter=50, maxtime=10 ** 6, maxsample=10000)
            ts.append(time.perf_counter() - t0)
        mx["config1_branin_N50"] = {"N": 50, "d": 2, "maxiter": 50, "wall_ms": 1e3 * min(ts), "nsamples": cdirectGP.last["nsamples"], "opt": opt}
        line["maximizeEI_wall_ms"] = mx
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(wl)
        print(json.dumps(line))
    if dist is not None:
        L.ibo_comm_destroy()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
