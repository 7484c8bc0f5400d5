"""Timing of the batch expected improvement on one GPU: ibo_qei with and without the gradient for SE-ARD models with d = 6,
N in {2048, 8192}, B q = 2^16 points, q in {4, 16}, S in {256, 2048}; beside each N, ibo_score_grad (EI, libm arithmetic) on the
same 2^16 points; and maximizeQEI(q = 8) at N = 2048, d = 6.

Per call: warm-up calls, then the median of several, timed with CUDA events on the model's stream (ibo_stream_mark /
ibo_stream_elapsed_ms around the whole call, which ends in a stream synchronisation), and the kernel launches per call
(ibo_launch_count).  The GPU's name and power limit are read in the same run.  One JSON line per record on stdout (and appended to
--out).

    python tools/qei_timing.py --out qei_timing.json
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
from grad_timing import THETA, emit, gpu_info, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, nargs="+", default=[2048, 8192])
    ap.add_argument("--q", type=int, nargs="+", default=[4, 16])
    ap.add_argument("--S", type=int, nargs="+", default=[256, 2048])
    ap.add_argument("--points", type=int, default=1 << 16)
    ap.add_argument("--no-maximize", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    L = _lib.lib()
    _lib.require_gpu()
    info = gpu_info()
    d = 6
    rs = np.random.RandomState(0)
    for N in a.N:
        X = rs.rand(N, d)
        Y = np.sin(3 * X).sum(axis=1)
        m = _lib.Model(_lib.KERNEL_SE_ARD, THETA, X, Y, 0.1)
        h = m.handle
        ymax = float(Y.max())
        P = np.ascontiguousarray(rs.rand(a.points, d))
        M = a.points
        sc, dsc = np.empty(M), np.empty((M, d))
        grad_call = lambda: _lib.check(L.ibo_score_grad(h, _lib.dptr(P), M, _lib.ACQ_EI, ymax, 0.01, 0,  # noqa: E731
                                                        _lib.dptr(sc), _lib.dptr(dsc)))
        sg_dev, _, sg_launch = timed(L, h, grad_call, 2, 5)
        for q in a.q:
            B = M // q
            for S in a.S:
                Z = np.ascontiguousarray(np.random.default_rng(S).standard_normal((q, S)))
                vals, dv, vals0 = np.empty(B), np.empty((B, q, d)), np.empty(B)
                nbad = ctypes.c_int(0)
                call_g = lambda: _lib.check(L.ibo_qei(h, _lib.dptr(P), B, q, _lib.dptr(Z), S, ymax, 0.01, 0.0,  # noqa: E731
                                                      _lib.dptr(vals), _lib.dptr(dv), ctypes.byref(nbad)))
                call_v = lambda: _lib.check(L.ibo_qei(h, _lib.dptr(P), B, q, _lib.dptr(Z), S, ymax, 0.01, 0.0,  # noqa: E731
                                                      _lib.dptr(vals0), None, ctypes.byref(nbad)))
                g_dev, g_wall, g_launch = timed(L, h, call_g, 2, 5)
                v_dev, v_wall, v_launch = timed(L, h, call_v, 2, 5)
                assert np.array_equal(vals, vals0) and nbad.value == 0
                emit(dict(kind="qei", N=N, d=d, B=B, q=q, S=S, points=M, kernel="se_ard", noise=0.1,
                          qei_grad_ms_device=g_dev, qei_grad_ms_wall=g_wall, qei_grad_launches=g_launch,
                          qei_value_ms_device=v_dev, qei_value_ms_wall=v_wall, qei_value_launches=v_launch,
                          score_grad_ms_device=sg_dev, score_grad_launches=sg_launch, qei_grad_over_score_grad=g_dev / sg_dev,
                          mean_value=float(np.mean(vals)), **info), a.out)
        m.close()
    if a.no_maximize:
        return
    from ibo_b200.acquisition import maximizeQEI, thompsonBatch
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    r = np.random.RandomState(5)
    X = r.rand(2048, d)
    gp = GaussianProcess(GaussianKernel_ard(THETA), X, np.sin(2 * X).sum(axis=1), noise=0.1)
    bounds = [[0., 1.]] * d
    res = []
    for _ in range(2):                                    # the first warms up
        t0 = time.perf_counter()
        val, batch = maximizeQEI(gp, bounds, 8, samples=512, seed=0, starts=8)
        res.append(1e3 * (time.perf_counter() - t0))
    t0 = time.perf_counter()
    for k in range(8):
        thompsonBatch(gp, bounds, 8, seed=k)
    t_starts = 1e3 * (time.perf_counter() - t0)
    last = maximizeQEI.last
    emit(dict(kind="maximizeQEI", N=2048, d=d, q=8, samples=512, starts=8, wall_ms=res[-1], thompson_starts_ms=t_starts,
              evaluations=last["evaluations"], value=val, best_start_value=float(np.max(last["start_values"])), **info), a.out)


if __name__ == "__main__":
    main()
