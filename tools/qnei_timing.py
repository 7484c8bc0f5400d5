"""Timing of the noisy batch expected improvement on one GPU: ibo_qnei with and without the gradient beside ibo_qei (values and
gradient) on the same 2^16 points, for SE-ARD models with d = 6, N in {2048, 8192}, P in {256, N} (the baseline: the first P
training points), q in {4, 16}, S in {256, 1024}; and maximizeQNEI(q = 8) at N = 2048, d = 6 with the default baseline.

Per call: two warm-up calls, then the median of five, timed with CUDA events on the model's stream (tools/grad_timing.timed), and
the kernel launches per call.  The GPU's name, power limit and max SM clock are read in the same run.  --profile (a run of its own):
torch.profiler's kernel times of the dense GEMM (gemm_kernel: C, H, Tbar, U) and of the triangular GEMMs (trimm_kernel /
trimm_t_kernel: V, T, Cbar, y) in one ibo_qnei call with the gradient, the dense GEMMs' FLOPs from the shapes, and their rate as a
share of the FP64 DMMA peak that ibo_fp64_peak measures on the same GPU.  One JSON line per record on stdout (and appended to --out).

    python tools/qnei_timing.py --out qnei_timing.json
    python tools/qnei_timing.py --profile --no-maximize --out qnei_timing.json
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


def r128(x):
    return (x + 127) // 128 * 128


def dense_gemm_flop(N, P, S, B, q, grad):
    """FLOPs of the dense GEMMs of one ibo_qnei call: C = K - V_b^T V_q (Pp x Np x Mcp), H = Z_b^T T (Sp x Pp x Mcp) and, with the
    gradient, Tbar = Z_b E (Pp x Sp x Mcp) and U += V_b Cbar / 2 (Np x Pp x Mcp), chunk by chunk"""
    Np, Pp, Sp = r128(N), r128(P), r128(S)
    pts = max(128, (1 << 26) // (2 * Np + 2 * Pp + Sp) // 128 * 128)
    Bc = pts // q
    flop = 0.0
    for b0 in range(0, B, Bc):
        Mcp = r128(min(Bc, B - b0) * q)
        f = Pp * Np + Sp * Pp
        if grad:
            f += Pp * Sp + Np * Pp
        flop += 2.0 * f * Mcp
    return flop


def profile_call(call):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    us = {}
    total = 0.0
    for e in prof.events():
        if e.device_time <= 0:
            continue
        total += e.device_time
        for k in ("gemm_kernel", "trimm_t_kernel", "trimm_kernel"):
            if k in e.name:
                us[k] = us.get(k, 0.0) + e.device_time
                break
    return us, total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, nargs="+", default=[2048, 8192])
    ap.add_argument("--P", nargs="+", default=["256", "N"])
    ap.add_argument("--q", type=int, nargs="+", default=[4, 16])
    ap.add_argument("--S", type=int, nargs="+", default=[256, 1024])
    ap.add_argument("--points", type=int, default=1 << 16)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--no-maximize", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    L = _lib.lib()
    _lib.require_gpu()
    info = gpu_info()
    peak = ctypes.c_double(0)
    if a.profile:
        _lib.check(L.ibo_fp64_peak(0, ctypes.byref(peak)))
    d = 6
    rs = np.random.RandomState(0)
    jitter = 1e-8
    for N in a.N:
        X = rs.rand(N, d)
        Y = np.sin(3 * X).sum(axis=1)
        m = _lib.Model(_lib.KERNEL_SE_ARD, THETA, X, Y, 0.1)
        h = m.handle
        ymax = float(Y.max())
        Pts = np.ascontiguousarray(rs.rand(a.points, d))
        M = a.points
        for q in a.q:
            B = M // q
            for S in a.S:
                Zq = np.ascontiguousarray(np.random.default_rng(S).standard_normal((q, S)))
                qv, qg = np.empty(B), np.empty((B, q, d))
                nbad, info_ = ctypes.c_int(0), ctypes.c_int(0)
                qei_g = lambda: _lib.check(L.ibo_qei(h, _lib.dptr(Pts), B, q, _lib.dptr(Zq), S, ymax, 0.01, 0.0,  # noqa: E731
                                                     _lib.dptr(qv), _lib.dptr(qg), ctypes.byref(nbad)))
                qei_v = lambda: _lib.check(L.ibo_qei(h, _lib.dptr(Pts), B, q, _lib.dptr(Zq), S, ymax, 0.01, 0.0,  # noqa: E731
                                                     _lib.dptr(qv), None, ctypes.byref(nbad)))
                ei_g_dev, _, ei_g_launch = timed(L, h, qei_g, 2, 5)
                ei_v_dev, _, ei_v_launch = timed(L, h, qei_v, 2, 5)
                for Ps in a.P:
                    P = N if Ps == "N" else int(Ps)
                    Xbase = np.ascontiguousarray(X[:P])
                    Z = np.ascontiguousarray(np.random.default_rng(S + P).standard_normal((P + q, S)))
                    vals, dv, vals0, inc = np.empty(B), np.empty((B, q, d)), np.empty(B), np.empty(S)
                    call_g = lambda: _lib.check(L.ibo_qnei(h, _lib.dptr(Pts), B, q, _lib.dptr(Xbase), P, _lib.dptr(Z), S,  # noqa: E731
                                                           jitter, _lib.dptr(vals), _lib.dptr(dv), _lib.dptr(inc),
                                                           ctypes.byref(nbad), ctypes.byref(info_)), info_.value)
                    call_v = lambda: _lib.check(L.ibo_qnei(h, _lib.dptr(Pts), B, q, _lib.dptr(Xbase), P, _lib.dptr(Z), S,  # noqa: E731
                                                           jitter, _lib.dptr(vals0), None, None,
                                                           ctypes.byref(nbad), ctypes.byref(info_)), info_.value)
                    if a.profile:
                        call_g()
                        us, total = profile_call(call_g)
                        flop = dense_gemm_flop(N, P, S, B, q, True)
                        rec = dict(kind="qnei_profile", N=N, P=P, q=q, S=S, points=M, d=d, dense_gemm_flop=flop,
                                   kernel_ms_total=total * 1e-3, fp64_peak_tflops=peak.value, **info)
                        for k, t in us.items():
                            rec[k + "_ms"] = t * 1e-3
                            rec[k + "_share_of_call"] = t / total
                        if "gemm_kernel" in us:
                            tf = flop / (us["gemm_kernel"] * 1e-6) / 1e12
                            rec["gemm_kernel_tflops"] = tf
                            rec["gemm_kernel_share_of_peak"] = tf / peak.value
                        emit(rec, a.out)
                        continue
                    g_dev, g_wall, g_launch = timed(L, h, call_g, 2, 5)
                    v_dev, v_wall, v_launch = timed(L, h, call_v, 2, 5)
                    assert np.array_equal(vals, vals0) and nbad.value == 0
                    emit(dict(kind="qnei", N=N, P=P, d=d, B=B, q=q, S=S, points=M, kernel="se_ard", noise=0.1, jitter=jitter,
                              qnei_grad_ms_device=g_dev, qnei_grad_ms_wall=g_wall, qnei_grad_launches=g_launch,
                              qnei_value_ms_device=v_dev, qnei_value_ms_wall=v_wall, qnei_value_launches=v_launch,
                              qei_grad_ms_device=ei_g_dev, qei_grad_launches=ei_g_launch,
                              qei_value_ms_device=ei_v_dev, qei_value_launches=ei_v_launch,
                              value_over_qei=v_dev / ei_v_dev, grad_over_qei=g_dev / ei_g_dev,
                              mean_value=float(np.mean(vals)), **info), a.out)
        m.close()
    if a.no_maximize:
        return
    from ibo_b200.acquisition import maximizeQNEI, thompsonBatch
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    r = np.random.RandomState(5)
    X = r.rand(2048, d)
    gp = GaussianProcess(GaussianKernel_ard(THETA), X, np.sin(2 * X).sum(axis=1), noise=0.1)
    bounds = [[0., 1.]] * d
    res = []
    for _ in range(2):                                    # the first warms up
        t0 = time.perf_counter()
        val, batch = maximizeQNEI(gp, bounds, 8, samples=512, seed=0, starts=8)
        res.append(1e3 * (time.perf_counter() - t0))
    t0 = time.perf_counter()
    for k in range(8):
        thompsonBatch(gp, bounds, 8, seed=k, jitter=1e-8)
    t_starts = 1e3 * (time.perf_counter() - t0)
    last = maximizeQNEI.last
    emit(dict(kind="maximizeQNEI", N=2048, d=d, q=8, P=len(last["baseline"]), samples=512, starts=8, wall_ms=res[-1],
              thompson_starts_ms=t_starts, evaluations=last["evaluations"], value=val,
              best_start_value=float(np.max(last["start_values"])), **info), a.out)


if __name__ == "__main__":
    main()
