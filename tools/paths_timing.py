"""Timing of pathwise posterior samples on one GPU, for SE-ARD models with d = 6 and N in {2048, 8192}: ibo_paths_eval (values and
per-path argmax) over M = 2^20 candidates from host buffers for S in {16, 64, 128} and F in {1024, 4096}, plus the headline shape
N = 2048, S = 64, F = 2048; ibo_paths_create timed separately.  Beside them, in the same run: one EI pass over the same candidates on
the default path and with IBO_FLAG_FP64, and ibo_posterior_sample at M = 8192 and 16384 with the same S.

Per call: 2 warm-up calls, then the median of 5.  ibo_paths_eval and ibo_paths_create run on the paths' own stream and end in a stream
synchronisation, so they are timed by the host clock around the call (`ms_wall`); the EI passes and ibo_posterior_sample also get CUDA
events on the model's stream (`ms_device`).  Rates count the FP64 pipe's multiply-adds from the shapes, 2 N (d + S) + 2 F (d + S) flop
per candidate (distances or phases, then the product with the coefficients); the exp and cos counts are listed apart.  The GPU's name,
power limit and the live FP64 tensor-pipe peak are read in the same run.  One JSON line per record on stdout (and appended to --out).

    python tools/paths_timing.py --out profiles/r07_paths_timing.json
"""
import argparse
import ctypes
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from ibo_b200 import _lib  # noqa: E402
from ibo_b200.gaussianprocess import path_draws  # noqa: E402
from grad_timing import THETA, emit, gpu_info, timed  # noqa: E402


def wall(call, warmup, reps):
    for _ in range(warmup):
        call()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        call()
        t.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(t))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, nargs="+", default=[2048, 8192])
    ap.add_argument("--M", type=int, default=1 << 20)
    ap.add_argument("--S", type=int, nargs="+", default=[16, 64, 128])
    ap.add_argument("--F", type=int, nargs="+", default=[1024, 4096])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    L = _lib.lib()
    _lib.require_gpu()
    info = gpu_info()
    peak = ctypes.c_double(0)
    _lib.check(L.ibo_fp64_peak(0, ctypes.byref(peak)))
    info["fp64_peak_tflops"] = peak.value
    d, M = 6, a.M
    rs = np.random.RandomState(0)
    p = _lib.dptr
    P = np.ascontiguousarray(rs.rand(M, d))
    for N in a.N:
        X = rs.rand(N, d)
        Y = np.sin(3 * X).sum(axis=1)
        m = _lib.Model(_lib.KERNEL_SE_ARD, THETA, X, Y, 0.1)
        h = m.handle
        ei = {}
        sc, best, bidx = np.empty(M), ctypes.c_double(0), ctypes.c_long(0)
        for path, fl in (("default", 0), ("fp64", _lib.FLAG_FP64)):
            call = lambda: _lib.check(L.ibo_score_batch(h, p(P), M, _lib.ACQ_EI, float(Y.max()), 0.01, fl, p(sc), None, None,  # noqa: E731
                                                        ctypes.byref(best), ctypes.byref(bidx)))
            ei[path] = timed(L, h, call, 2, 5)[:2]
        joint = {}
        shapes = [(S, F) for S in a.S for F in a.F]
        if N == 2048:
            shapes.append((64, 2048))
        for S, F in shapes:
            dr = path_draws(_lib.KERNEL_SE_ARD, d, F, S, N, seed=S + F)
            t0 = time.perf_counter()
            paths = m.sample_paths(*dr)
            create_first = 1e3 * (time.perf_counter() - t0)
            create_ms = wall(lambda: m.sample_paths(*dr).close(), 1, 3)
            vals = np.empty((M, S))
            bst, idx = np.empty(S), np.empty(S, dtype=np.int64)
            ev = lambda: _lib.check(L.ibo_paths_eval(paths._h, p(P), M, p(vals), p(bst), idx.ctypes.data_as(ctypes.POINTER(ctypes.c_long))))  # noqa: E731
            ev_arg = lambda: _lib.check(L.ibo_paths_eval(paths._h, p(P), M, None, p(bst), idx.ctypes.data_as(ctypes.POINTER(ctypes.c_long))))  # noqa: E731
            t_vals = wall(ev, 2, 5)
            t_arg = wall(ev_arg, 2, 5)
            flop = float(M) * (2 * N * (d + S) + 2 * F * (d + S))
            rec = dict(kind="paths_eval", N=N, d=d, M=M, S=S, F=F, flop_fp64_pipe=flop, exp_count=float(M) * N, cos_count=float(M) * F,
                       eval_ms_wall=t_vals, eval_argmax_only_ms_wall=t_arg,
                       tflops=flop / t_arg * 1e-9, share_of_fp64_peak=flop / t_arg * 1e-9 / peak.value,
                       create_ms_wall=create_ms, create_first_ms_wall=create_first,
                       ei_default_ms_device=ei["default"][0], ei_default_ms_wall=ei["default"][1],
                       ei_fp64_ms_device=ei["fp64"][0], ei_fp64_ms_wall=ei["fp64"][1],
                       argmax_only_over_ei_fp64=t_arg / ei["fp64"][1], argmax_only_over_ei_default=t_arg / ei["default"][1], **info)
            for Mj in (8192, 16384):
                if (S, Mj) in joint:
                    rec.update(joint[S, Mj])
                    continue
                Z = np.random.default_rng(Mj).standard_normal((Mj, S))
                am = np.empty(S, dtype=np.int64)
                info_c = ctypes.c_int(0)
                js = lambda: _lib.check(L.ibo_posterior_sample(h, p(P), Mj, p(Z), S, 0.0, None, am.ctypes.data_as(  # noqa: E731
                    ctypes.POINTER(ctypes.c_long)), ctypes.byref(info_c)))
                dev, wl, _ = timed(L, h, js, 2, 5)
                joint[S, Mj] = {"joint_sample_M%d_ms_device" % Mj: dev, "joint_sample_M%d_ms_wall" % Mj: wl}
                rec.update(joint[S, Mj])
            emit(rec, a.out)
            paths.close()
        m.close()


if __name__ == "__main__":
    main()
