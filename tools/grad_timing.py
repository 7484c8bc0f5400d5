"""Timing of the candidate gradients on one GPU: ibo_score_grad (EI, libm arithmetic) next to ibo_score_batch with IBO_FLAG_FP64 on the
same candidates, for SE-ARD models with d = 6, N in {2048, 8192}, M in {64, 2^16, 2^20}; and maximizeEI with polish=8 against
plain maximizeEI at N = 2048, d = 6 and at config #5's shape (N = 4096, d = 20, 200 DIRECT iterations).

Per call: warm-up calls, then the median of several, timed two ways -- CUDA events on the model's stream (ibo_stream_mark /
ibo_stream_elapsed_ms around the call, which ends in a stream synchronisation) and the host wall clock -- and the kernel launches
per call (ibo_launch_count).  With --profile, one extra pass per N at M = 2^16 runs under torch.profiler (CUDA activities) for the
time of the two triangular GEMM kernels (trimm_kernel: V = W K*, trimm_t_kernel: Z = W^T V); their FLOPs are counted from the
tile shapes (2 * 128^3 per 128 x 128 x 128 tile step, nb (nb + 1) / 2 steps per column tile) and set against the live
ibo_fp64_peak.  The GPU's name and power limit are read in the same run.  One JSON line per record on stdout (and appended to
--out).

    python tools/grad_timing.py --profile --out grad_timing.json
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


def timed(L, h, call, warmup, reps):
    for _ in range(warmup):
        call()
    dev, wall, launches = [], [], []
    ms = ctypes.c_float(0)
    for _ in range(reps):
        n0 = L.ibo_launch_count()
        _lib.check(L.ibo_stream_mark(h, 0))
        t0 = time.perf_counter()
        call()
        t1 = time.perf_counter()
        _lib.check(L.ibo_stream_mark(h, 1))
        _lib.check(L.ibo_stream_elapsed_ms(h, ctypes.byref(ms)))
        launches.append(L.ibo_launch_count() - n0)
        dev.append(ms.value)
        wall.append(1e3 * (t1 - t0))
    return float(np.median(dev)), float(np.median(wall)), int(np.median(launches))


def emit(rec, out):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "a") as f:
            f.write(line + "\n")


def gemm_profile(m, Xs, N):
    """kernel times of the two W GEMMs in one ibo_score_grad call, from torch.profiler"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    M = Xs.shape[0]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.score_grad(Xs, _lib.ACQ_EI, 0.0, 0.01, _lib.FLAG_MODE_CPP)
        torch.cuda.synchronize()
    us = {}
    for e in prof.events():
        for k in ("trimm_t_kernel", "trimm_kernel"):
            if k in e.name:
                us[k] = us.get(k, 0.0) + e.device_time
                break
    Np = (N + 127) // 128 * 128
    nb = Np // 128
    chunk = max(128, (512 << 20) // (16 * Np) // 128 * 128)
    cols = 0
    for c0 in range(0, M, chunk):
        cols += (min(chunk, M - c0) + 127) // 128
    flop = 2.0 * 128 ** 3 * cols * nb * (nb + 1) / 2        # per GEMM
    return us, flop


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, nargs="+", default=[2048, 8192])
    ap.add_argument("--M", type=int, nargs="+", default=[64, 1 << 16, 1 << 20])
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--no-direct", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    L = _lib.lib()
    _lib.require_gpu()
    info = gpu_info()
    peak = ctypes.c_double(0)
    _lib.check(L.ibo_fp64_peak(0, ctypes.byref(peak)))
    d = 6
    rs = np.random.RandomState(0)
    for N in a.N:
        X = rs.rand(N, d)
        Y = np.sin(3 * X).sum(axis=1)
        m = _lib.Model(_lib.KERNEL_SE_ARD, THETA, X, Y, 0.1)
        h = m.handle
        ymax = float(Y.max())
        for M in a.M:
            Xs = np.ascontiguousarray(rs.rand(M, d))
            sc, dsc, sb = np.empty(M), np.empty((M, d)), np.empty(M)
            grad_call = lambda: _lib.check(L.ibo_score_grad(h, _lib.dptr(Xs), M, _lib.ACQ_EI, ymax, 0.01, 0,  # noqa: E731
                                                            _lib.dptr(sc), _lib.dptr(dsc)))
            best, bidx = ctypes.c_double(0), ctypes.c_long(0)
            score_call = lambda: _lib.check(L.ibo_score_batch(h, _lib.dptr(Xs), M, _lib.ACQ_EI, ymax, 0.01, _lib.FLAG_FP64,  # noqa: E731
                                                              _lib.dptr(sb), None, None, ctypes.byref(best), ctypes.byref(bidx)))
            warm, reps = (3, 21) if M <= 4096 else ((2, 5) if M <= (1 << 16) else (1, 2))
            g_dev, g_wall, g_launch = timed(L, h, grad_call, warm, reps)
            s_dev, s_wall, s_launch = timed(L, h, score_call, warm, reps)
            assert np.array_equal(sc, sb)
            emit(dict(kind="call", N=N, M=M, d=d, kernel="se_ard", acq="ei", noise=0.1,
                      grad_ms_device=g_dev, grad_ms_wall=g_wall, grad_launches=g_launch, grad_cands_per_s=M / (g_dev * 1e-3),
                      score_fp64_ms_device=s_dev, score_fp64_ms_wall=s_wall, score_fp64_launches=s_launch,
                      score_fp64_cands_per_s=M / (s_dev * 1e-3), grad_over_score=g_dev / s_dev, **info), a.out)
            if a.profile and M == (1 << 16):
                us, flop = gemm_profile(m, Xs, N)
                rec = dict(kind="gemm", N=N, M=M, d=d, flop_per_gemm=flop, fp64_peak_tflops=peak.value, **info)
                for k, t in us.items():
                    rec[k + "_ms"] = t * 1e-3
                    rec[k + "_tflops"] = flop / (t * 1e-6) / 1e12
                    rec[k + "_share_of_peak"] = flop / (t * 1e-6) / 1e12 / peak.value
                emit(rec, a.out)
        m.close()
    if a.no_direct:
        return
    from ibo_b200.acquisition import cdirectGP, maximizeEI
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    for N, dd, theta, iters in ((2048, 6, THETA, 50), (4096, 20, [1.0] * 20, 200)):
        r = np.random.RandomState(5)
        X = r.rand(N, dd)
        Y = np.sin(2 * X).sum(axis=1)
        gp = GaussianProcess(GaussianKernel_ard(theta), X, Y, noise=0.1)
        bounds = [[0., 1.]] * dd
        res = {}
        for polish in (0, 8, 0, 8):            # alternating; the first of each warms up
            t0 = time.perf_counter()
            opt, optx = maximizeEI(gp, bounds, xi=0.01, maxiter=iters, maxtime=10 ** 6, maxsample=10 ** 9, polish=polish)
            t = 1e3 * (time.perf_counter() - t0)
            res[polish] = dict(wall_ms=t, opt=float(opt), polish=cdirectGP.last.get("polish"), nsamples=cdirectGP.last["nsamples"])
        fp64 = _lib.FLAG_MODE_CPP | _lib.FLAG_FP64
        emit(dict(kind="maximizeEI", N=N, d=dd, maxiter=iters, plain_ms=res[0]["wall_ms"], polish8_ms=res[8]["wall_ms"],
                  plain_opt=res[0]["opt"], polish8_opt=res[8]["opt"], polish=res[8]["polish"], nsamples=res[0]["nsamples"],
                  arithmetic="libm (IBO_FLAG_MODE_CPP); polished value in FP64 (%d)" % fp64, **info), a.out)


if __name__ == "__main__":
    main()
