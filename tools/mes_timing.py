"""Timing of max-value entropy search on one GPU, for SE-ARD models with d = 6 and N in {2048, 8192}: ibo_mes values at M in
{2^16, 2^20} and K in {10, 100} on the default path and with IBO_FLAG_FP64, ibo_mes with the gradient at M = 2^16, and
ibo_max_value_gumbel at M in {2^16, 2^20}; beside them, on the same points and path, ibo_score_batch (EI), ibo_posterior_batch and
ibo_score_grad (EI).  Then maximizeMES wall time at N = 2048, d = 6 and at config #1's shape (Branin, N = 50, d = 2).

Per call: 2 warm-up calls, then the median of 5, timed with CUDA events on the model's stream (ibo_stream_mark /
ibo_stream_elapsed_ms around the whole call from host buffers, which ends in a stream synchronisation).  The GPU's name and power
limit are read in the same run.  One JSON line per record on stdout (and appended to --out).

    python tools/mes_timing.py --out mes_timing.json
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
    ap.add_argument("--M", type=int, nargs="+", default=[1 << 16, 1 << 20])
    ap.add_argument("--K", type=int, nargs="+", default=[10, 100])
    ap.add_argument("--no-maximize", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    L = _lib.lib()
    _lib.require_gpu()
    info = gpu_info()
    d = 6
    rs = np.random.RandomState(0)
    p = _lib.dptr
    for N in a.N:
        X = rs.rand(N, d)
        Y = np.sin(3 * X).sum(axis=1)
        m = _lib.Model(_lib.KERNEL_SE_ARD, THETA, X, Y, 0.1)
        h = m.handle
        ymax = float(Y.max())
        for M in a.M:
            P = np.ascontiguousarray(rs.rand(M, d))
            q, loc, scale = np.empty(3), ctypes.c_double(0), ctypes.c_double(0)
            gum = lambda: _lib.check(L.ibo_max_value_gumbel(h, p(P), M, 0, p(q), ctypes.byref(loc), ctypes.byref(scale)))  # noqa: E731
            gum_dev, gum_wall, gum_launch = timed(L, h, gum, 2, 5)
            mu, s2 = np.empty(M), np.empty(M)
            for path, fl in (("default", 0), ("fp64", _lib.FLAG_FP64)):
                post = lambda: _lib.check(L.ibo_posterior_batch(h, p(P), M, fl, p(mu), p(s2)))  # noqa: E731
                post_dev, _, _ = timed(L, h, post, 2, 5)
                sc, best, bidx = np.empty(M), ctypes.c_double(0), ctypes.c_long(0)
                ei = lambda: _lib.check(L.ibo_score_batch(h, p(P), M, _lib.ACQ_EI, ymax, 0.01, fl, p(sc), None, None,  # noqa: E731
                                                          ctypes.byref(best), ctypes.byref(bidx)))
                ei_dev, _, _ = timed(L, h, ei, 2, 5)
                if path == "default":
                    emit(dict(kind="gumbel", N=N, d=d, M=M, path=path, gumbel_ms_device=gum_dev, gumbel_ms_wall=gum_wall,
                              gumbel_launches=gum_launch, posterior_ms_device=post_dev, gumbel_over_posterior=gum_dev / post_dev,
                              loc=loc.value, scale=scale.value, **info), a.out)
                for K in a.K:
                    u = np.random.default_rng(K).uniform(0.01, 0.99, K)
                    ys = np.ascontiguousarray(loc.value - scale.value * np.log(-np.log(u)))
                    vals = np.empty(M)
                    mes = lambda: _lib.check(L.ibo_mes(h, p(P), M, p(ys), K, fl, p(vals), None,  # noqa: E731
                                                       ctypes.byref(best), ctypes.byref(bidx)))
                    v_dev, v_wall, v_launch = timed(L, h, mes, 2, 5)
                    rec = dict(kind="mes", N=N, d=d, M=M, K=K, path=path, mes_ms_device=v_dev, mes_ms_wall=v_wall,
                               mes_launches=v_launch,
                               ei_ms_device=ei_dev, posterior_ms_device=post_dev, mes_over_ei=v_dev / ei_dev,
                               mean_value=float(np.mean(vals)), **info)
                    if M == min(a.M) and path == "default":
                        dv, sg, dsg = np.empty((M, d)), np.empty(M), np.empty((M, d))
                        mg = lambda: _lib.check(L.ibo_mes(h, p(P), M, p(ys), K, 0, p(vals), p(dv),  # noqa: E731
                                                          ctypes.byref(best), ctypes.byref(bidx)))
                        g_dev, g_wall, g_launch = timed(L, h, mg, 2, 5)
                        sgc = lambda: _lib.check(L.ibo_score_grad(h, p(P), M, _lib.ACQ_EI, ymax, 0.01, 0, p(sg), p(dsg)))  # noqa: E731
                        sg_dev, _, _ = timed(L, h, sgc, 2, 5)
                        rec.update(mes_grad_ms_device=g_dev, mes_grad_ms_wall=g_wall, mes_grad_launches=g_launch,
                                   score_grad_ms_device=sg_dev, mes_grad_over_score_grad=g_dev / sg_dev)
                    emit(rec, a.out)
        m.close()
    if a.no_maximize:
        return
    from ibo_b200.acquisition import maximizeMES
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    from ibo_b200.utils.latinhypercube import lhcSample
    r = np.random.RandomState(5)
    X = r.rand(2048, d)
    shapes = [("N2048_d6", GaussianProcess(GaussianKernel_ard(THETA), X, np.sin(2 * X).sum(axis=1), noise=0.1), [[0., 1.]] * d)]
    bb = [[-5., 10.], [0., 15.]]                          # config #1: demo.py-style Branin, N = 50, SE-ARD [3.4, 10]
    Xb = np.array(lhcSample(bb, 50, seed=0))
    Yb = -((Xb[:, 1] - (5.1 / (4 * np.pi ** 2)) * Xb[:, 0] ** 2 + 5 * Xb[:, 0] / np.pi - 6) ** 2
           + 10 * (1 - 1 / (8 * np.pi)) * np.cos(Xb[:, 0]) + 10) / 100.0
    shapes.append(("config1_branin_N50", GaussianProcess(GaussianKernel_ard([3.4, 10.0]), Xb, Yb, noise=0.1), bb))
    for name, gp, bounds in shapes:
        for polish in (0, 8):
            res = []
            for _ in range(3):                            # the first warms up
                t0 = time.perf_counter()
                opt, optx = maximizeMES(gp, bounds, n_samples=10, seed=0, maxiter=50, maxtime=10 ** 6, polish=polish)
                res.append(1e3 * (time.perf_counter() - t0))
            last = maximizeMES.last
            emit(dict(kind="maximizeMES", shape=name, N=len(gp.Y), d=len(bounds), maxiter=50, n_samples=10, candidates=16384,
                      polish=polish, wall_ms=float(np.median(res[1:])), direct_samples=last["samples"],
                      polish_evaluations=None if last["polish"] is None else last["polish"]["evaluations"], opt=opt, **info), a.out)


if __name__ == "__main__":
    main()
