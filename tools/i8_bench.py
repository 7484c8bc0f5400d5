"""Times the INT8 wide-batch path against the FP64 DMMA path on resident candidates (device time of ibo_score_resident):
   python tools/i8_bench.py [N d M kind]      kind: se | m5 (Matern-5/2 ARD)
Prints evals/s of both paths, the K1 / K2 / K3 split (IBO_FLAG_PROFILE runs the chunks back to back), the live INT8 peak and the
agreement of the two paths."""
import ctypes
import sys

import numpy as np

sys.path.insert(0, __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__))))
from ibo_b200 import _lib
from ibo_b200.gaussianprocess import GaussianProcess
from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard, MaternKernel5_ard

N = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
d = int(sys.argv[2]) if len(sys.argv) > 2 else 6
M = int(sys.argv[3]) if len(sys.argv) > 3 else 1 << 20
kind = sys.argv[4] if len(sys.argv) > 4 else "se"
rs = np.random.RandomState(0)
X = rs.rand(N, d); Y = np.sin(2 * X).sum(axis=1)
theta = [0.5 + 0.05 * j for j in range(d)]
gp = GaussianProcess(MaternKernel5_ard(theta + [1.0]) if kind == "m5" else GaussianKernel_ard(theta), X, Y, noise=0.1)
m = gp.model
Xs = np.ascontiguousarray(np.random.RandomState(1).rand(M, d))
c = _lib.ResidentCandidates(m, Xs)
L = _lib.lib()
ymax = float(Y.max())
res = {}
for name, fl in (("fp64", _lib.FLAG_MODE_CPP | _lib.FLAG_FP64), ("int8", _lib.FLAG_MODE_CPP)):
    s = np.empty(M)
    b = c.score(_lib.ACQ_EI, ymax, 0.01, fl, scores_out=s)
    ts = [c.score(_lib.ACQ_EI, ymax, 0.01, fl)[2] for _ in range(3)]
    c.score(_lib.ACQ_EI, ymax, 0.01, fl | _lib.FLAG_PROFILE)
    p = m.profile()
    res[name] = (s, b, min(ts), p)
    print("%s: %.3f ms  %.2f M evals/s   K1 %.2f  K2 %.2f  K3 %.2f ms (profiled back to back)  argmax %d  guarded %d"
          % (name, min(ts), M / min(ts) / 1e3, p["k1_ms"], p["k2_ms"], p["k3_ms"], b[1], m.last_guarded()), flush=True)
_lib.set_option("i8_pipe", 0)
ts = [c.score(_lib.ACQ_EI, ymax, 0.01, _lib.FLAG_MODE_CPP)[2] for _ in range(3)]
_lib.set_option("i8_pipe", 1)
print("int8 without the two-stream pipeline: %.3f ms" % min(ts))
pk, pks = ctypes.c_double(0), ctypes.c_double(0)
_lib.check(L.ibo_i8_peak2(0, 2.0, ctypes.byref(pk), ctypes.byref(pks)))
nb = (N + 127) // 128
ops = 2.0 * 28 * 128 * 32 * 4 * (nb * (nb + 1) // 2)
k2 = res["int8"][3]["k2_ms"]
ach = M * ops / (k2 * 1e-3) / 1e12
print("K2 int8: %.2f TOP/s; burst peak %.2f (frac %.3f), sustained peak with random operands %.2f (frac %.3f)" % (ach, pk.value, ach / pk.value, pks.value, ach / pks.value))
a, b = res["fp64"][0], res["int8"][0]
print("max |dEI| / max(|EI|, 1e-5) = %.3g   same argmax %s   speed-up %.2fx"
      % (np.max(np.abs(a - b) / np.maximum(np.abs(a), 1e-5)), res["fp64"][1][1] == res["int8"][1][1], res["fp64"][2] / res["int8"][2]))
