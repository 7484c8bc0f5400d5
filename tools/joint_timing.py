"""Timing of the joint posterior on one GPU: ibo_posterior_cov and ibo_posterior_sample (F = NULL, only the S argmax indices
come back) for SE-ARD models with d = 6, N in {512, 2048, 8192}, M in {1024, 4096, 8192}, S = 128.

Per configuration and entry point: 2 warm-up calls, then the median of 5 calls, timed two ways -- CUDA events on the model's
stream (ibo_stream_mark / ibo_stream_elapsed_ms around the call; the window also covers the host part of the call, which ends
in a stream synchronisation) and the host wall clock.  FP64 work from shapes: V = W R(X, X*) is N^2 M, Sigma = R** - V^T V is
N M^2, the Cholesky of Sigma M^3 / 3 and the samples M^2 S; rates against the live ibo_fp64_peak.  The GPU's name and power
limit are read in the same run.  One JSON line per configuration on stdout (and appended to --out).

    python tools/joint_timing.py --out joint_timing.json
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from ibo_b200 import _lib  # noqa: E402

THETA = [.53, .57, 2.5, .34, .27, .35]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def timed(L, h, call, warmup=2, reps=5):
    for _ in range(warmup):
        call()
    dev, wall = [], []
    ms = ctypes.c_float(0)
    for _ in range(reps):
        _lib.check(L.ibo_stream_mark(h, 0))
        t0 = time.perf_counter()
        call()
        t1 = time.perf_counter()
        _lib.check(L.ibo_stream_mark(h, 1))
        _lib.check(L.ibo_stream_elapsed_ms(h, ctypes.byref(ms)))
        dev.append(ms.value)
        wall.append(1e3 * (t1 - t0))
    return float(np.median(dev)), float(np.median(wall))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, nargs="+", default=[512, 2048, 8192])
    ap.add_argument("--M", type=int, nargs="+", default=[1024, 4096, 8192])
    ap.add_argument("--S", type=int, default=128)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    L = _lib.lib()
    _lib.require_gpu()
    info = gpu_info()
    peak = ctypes.c_double(0)
    _lib.check(L.ibo_fp64_peak(0, ctypes.byref(peak)))
    d, S = 6, a.S
    rs = np.random.RandomState(0)
    for N in a.N:
        X = rs.rand(N, d)
        Y = np.sin(3 * X).sum(axis=1)
        m = _lib.Model(_lib.KERNEL_SE_ARD, THETA, X, Y, 0.1)
        h = m.handle
        for M in a.M:
            Xs = np.ascontiguousarray(rs.rand(M, d))
            Z = np.ascontiguousarray(np.random.default_rng(M).standard_normal((M, S)))
            mu, cov = np.empty(M), np.empty((M, M))
            am = np.empty(S, dtype=np.int64)
            info_c = ctypes.c_int(0)
            pl = am.ctypes.data_as(ctypes.POINTER(ctypes.c_long))
            cov_call = lambda: _lib.check(L.ibo_posterior_cov(h, _lib.dptr(Xs), M, _lib.dptr(mu), _lib.dptr(cov)))   # noqa: E731
            smp_call = lambda: _lib.check(L.ibo_posterior_sample(h, _lib.dptr(Xs), M, _lib.dptr(Z), S, 1e-9, None, pl,   # noqa: E731
                                                                 ctypes.byref(info_c)), info_c.value)
            cov_dev, cov_wall = timed(L, h, cov_call)
            smp_dev, smp_wall = timed(L, h, smp_call)
            fl_v, fl_sig, fl_chol, fl_smp = float(N) ** 2 * M, float(N) * M * M, float(M) ** 3 / 3, float(M) ** 2 * S
            fl_cov = fl_v + fl_sig
            fl_all = fl_cov + fl_chol + fl_smp
            rec = dict(N=N, M=M, S=S, d=d, kernel="se_ard", noise=0.1,
                       flop=dict(V=fl_v, Sigma=fl_sig, chol=fl_chol, samples=fl_smp),
                       cov_ms_device=cov_dev, cov_ms_wall=cov_wall,
                       sample_ms_device=smp_dev, sample_ms_wall=smp_wall,
                       cov_tflops=fl_cov / (cov_dev * 1e-3) / 1e12,
                       sample_tflops=fl_all / (smp_dev * 1e-3) / 1e12,
                       fp64_peak_tflops=peak.value,
                       cov_share_of_peak=fl_cov / (cov_dev * 1e-3) / 1e12 / peak.value,
                       sample_share_of_peak=fl_all / (smp_dev * 1e-3) / 1e12 / peak.value,
                       cov_bytes_to_host=8.0 * M * (M + 1), **info)
            line = json.dumps(rec)
            print(line, flush=True)
            if a.out:
                os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
                with open(a.out, "a") as f:
                    f.write(line + "\n")
        m.close()


if __name__ == "__main__":
    main()
