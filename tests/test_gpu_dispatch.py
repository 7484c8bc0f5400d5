"""Every template instance the scoring path (K1 -> K2 -> K3) can dispatch to, each against the FP64 oracle, and the options that are
documented to change no result bit (DESIGN section 4, "Determinism").

The instance lists at module level (DIMS, KERNEL_CLASSES, NARROW_MTS, ...) are checked against the dispatch code by
tests/test_dispatch_table.py on the CPU: a new bucket in score.cu / score_i8.cuh that no case here reaches fails the CPU suite.
Which K2 instance ran is not inferred from a port of the planner: option debug_plan makes the library print a line per latency-shape
plan ("[plan_narrow] ...") and per FP64 K2 launch ("[k2] ... MT=.. P1=.. DEEP=.."), and the `plans` fixture parses them.
Set DISPATCH_PLAN_LOG=<file> to keep every recorded line with the id of the test that produced it.

Bounds: 1e-10 relative on mu (floor 1e-3), on sigma^2 and on EI (floor 1e-5), as in tests/test_gpu_fuzz.py; the argmax is the
device's own maximum (lowest index on ties) and within the bound of the oracle's."""
import contextlib
import os
import re

import numpy as np
import pytest

from oracle import ibo_oracle as orc

pytestmark = pytest.mark.gpu

TOL = 1e-10
EI_FLOOR = 1e-5
XI = 0.01
NOISE = 0.1

# K1 instances: every d for every kernel class (template argument KC of kstar_mma_kernel / kstar_i8_kernel -> a kind that runs it;
# SE-iso shares class 0 with SE-ARD, Matern-5/2 class 2 with Matern-5/2-ARD)
DIMS = list(range(1, 41))
KERNEL_CLASSES = {0: orc.K_SE_ARD, 1: orc.K_MATERN3, 2: orc.K_MATERN5_ARD}
GUARD_DIMS = [21, 26, 32]                 # K1's cancellation guard at high d (with a prior: the P1 instances)
GRID_Z_BATCHES = [100, 200, 450, 1000, 2048]   # N = 2049: 1 / 2 / 4 / 8 / 16 K1 tiles -> grid.z = 16 / 8 / 4 / 2 / 1
# K2 latency shapes: trigemm_kernel<1, MT, P1, DEEP>
NARROW_MTS = [8, 4, 2, 1]
K2_DEEP = [0, 1]
K2_PRIOR = [False, True]
K2_NOBS = [129, 640, 2049, 100]           # 100: one row-block (with option tiny = 0)
K2_BATCHES = [1, 31, 33, 97, 2048]

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_CSRC = os.path.join(_ROOT, "ibo_b200", "csrc")


def _constant(fname, pattern):
    with open(os.path.join(_CSRC, fname)) as f:
        return float(re.search(pattern, f.read()).group(1))


CAND_INLINE = int(_constant("common.cuh", r"constexpr int CAND_INLINE = (\d+);"))        # doubles of K1's parameter-buffer batch
EXPAND_LIMIT = _constant("score.cu", r"constexpr double EXPAND_LIMIT = ([0-9.]+);")      # K1: |x|^2 + |y|^2 above it -> direct

# ------------------------------------------------------------------------------------------------------------------------------
# fixtures
# ------------------------------------------------------------------------------------------------------------------------------


@contextlib.contextmanager
def options(**kw):
    """set library options for the block, restore the previous values whatever happens"""
    from ibo_b200 import _lib
    old = {k: _lib.get_option(k) for k in kw}
    try:
        for k, v in kw.items():
            _lib.set_option(k, v)
        yield
    finally:
        for k, v in old.items():
            _lib.set_option(k, v)


_PLAN_RE = re.compile(r"\[plan_narrow\] nb=(\d+) ctaTiles=(\d+) -> MT=(\d+) G=(\d+) \((\d+) CTAs\)")
_K2_RE = re.compile(r"\[k2\] nb=(\d+) NT=(\d+) MT=(\d+) P1=(\d+) DEEP=(\d+) PDL=(\d+) grid=(\d+)x(\d+)")


class PlanRecorder(object):
    """debug_plan lines written to stderr since the last take()"""

    def __init__(self, capfd, nodeid):
        self.capfd, self.nodeid = capfd, nodeid
        self.log = os.environ.get("DISPATCH_PLAN_LOG")

    def take(self):
        err = self.capfd.readouterr().err
        plans = [dict(zip(("nb", "ctaTiles", "MT", "G", "CTAs"), map(int, g))) for g in _PLAN_RE.findall(err)]
        k2 = [dict(zip(("nb", "NT", "MT", "P1", "DEEP", "PDL", "gx", "gy"), map(int, g))) for g in _K2_RE.findall(err)]
        if self.log:
            with open(self.log, "a") as f:
                for line in err.splitlines():
                    if line.startswith("[plan_narrow]") or line.startswith("[k2]"):
                        f.write("%s\t%s\n" % (self.nodeid, line))
        return plans, k2

    def note(self, text):
        if self.log:
            with open(self.log, "a") as f:
                f.write("%s\t%s\n" % (self.nodeid, text))


@pytest.fixture
def plans(capfd, request):
    with options(debug_plan=1):
        rec = PlanRecorder(capfd, request.node.nodeid)
        rec.take()
        yield rec


# ------------------------------------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------------------------------------


def _rel(a, b, floor):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


def _hyper(kind, d, rs, scale):
    if kind in (orc.K_SE_ARD, orc.K_MATERN5_ARD):
        h = list(scale * (0.8 + 0.4 * rs.rand(d)))
        return h + [0.9] if kind == orc.K_MATERN5_ARD else h
    return [scale, 0.9]


def _problem(kind, d, N, M, seed, scale=None, near=1e-3, prior=False, noise=NOISE):
    """model data, a candidate pool with a third of it right next to training points (small sigma^2, k* far from 0), oracle"""
    from ibo_b200 import _lib
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    Y = np.sin(2.5 * X).sum(axis=1) + 0.1 * rs.randn(N)
    hyper = _hyper(kind, d, rs, 0.25 * np.sqrt(d) if scale is None else scale)
    pool = rs.rand(M, d)
    k = max(1, M // 3)
    idx = rs.choice(M, k, replace=False)
    theta = np.asarray(orc.KernelSpec(kind, hyper, d).theta)
    pool[idx] = X[rs.randint(N, size=k)] + near * theta * rs.randn(k, d)
    op = orc.PriorSpec(rs.rand(4, d), 0.3 * rs.randn(4), 0.5, np.zeros(d), np.ones(d)) if prior else None
    m = _lib.Model(kind, hyper, X, Y, noise, prior=op)
    o = orc.GPOracle(orc.KernelSpec(kind, hyper, d), X, Y, noise, prior=op)
    return m, o, X, Y, pool


def _assert_oracle(res, mu_o, s2_o, ymax, tag):
    sc, mu, s2, best, bidx = res
    assert _rel(mu, mu_o, 1e-3) <= TOL, tag
    assert _rel(s2, s2_o, 1e-300) <= TOL, tag
    want = orc.score(orc.ACQ_EI, "py", mu_o, s2_o, ymax, XI)
    assert _rel(sc, want, EI_FLOOR) <= TOL, tag
    assert best == sc[bidx] and bidx == int(np.argmax(sc)), tag
    assert want[bidx] >= want.max() - TOL * max(abs(want.max()), EI_FLOOR), tag


def _assert_close(a, b, tag):
    assert _rel(a[1], b[1], 1e-3) <= TOL and _rel(a[2], b[2], 1e-300) <= TOL and _rel(a[0], b[0], EI_FLOOR) <= TOL, tag


def _assert_same(a, b, tag):
    """scores, mu, sigma^2, best value and best index bit for bit"""
    for j, what in enumerate(("scores", "mu", "sigma^2")):
        if a[j] is not None or b[j] is not None:
            assert np.array_equal(a[j], b[j]), "%s: %s differ" % (tag, what)
    assert a[3] == b[3] and a[4] == b[4], "%s: best (%r, %d) vs (%r, %d)" % (tag, a[3], a[4], b[3], b[4])


def _score(m, Xs, ymax, flags=0, acq=orc.ACQ_EI, parm=XI):
    from ibo_b200 import _lib
    return m.score(np.ascontiguousarray(Xs), acq, ymax, parm, flags=_lib.FLAG_MODE_PY | flags, want_posterior=True)


# ------------------------------------------------------------------------------------------------------------------------------
# a. K1 instances
# ------------------------------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("kc", sorted(KERNEL_CLASSES))
@pytest.mark.parametrize("d", DIMS)
def test_k1_instance_matches_oracle(d, kc):
    """FP64 K1 kstar_mma_kernel<ceil(d/4), KC> (kstar_kernel beyond d = 32) on both sides of the parameter-buffer batch, INT8 K1
    kstar_i8_kernel<KC, DMAX(d)> on a wide batch, and option kstar_direct against the expansion"""
    from ibo_b200 import _lib
    kind = KERNEL_CLASSES[kc]
    N, Mw = 200, 2600
    m, o, X, Y, pool = _problem(kind, d, N, Mw, 1000 * kc + d)
    try:
        ymax = float(Y.max())
        mu_o, s2_o = o.posterior_batch(pool)
        ml = CAND_INLINE // d                      # ml * d <= CAND_INLINE < (ml + 1) * d
        runs = {}
        for M in (ml, ml + 1):
            runs["latency %d" % M] = (M, _score(m, pool[:M], ymax), _score(m, pool[:M], ymax, _lib.FLAG_FP64))
        wide_i8 = _score(m, pool, ymax)
        wide_fp = _score(m, pool, ymax, _lib.FLAG_FP64)
        with options(kstar_direct=1):
            direct = {M: _score(m, pool[:M], ymax) for M in (ml, ml + 1)}
            wide_direct = _score(m, pool, ymax, _lib.FLAG_FP64)
        tag = "kind %d d %d" % (kind, d)
        for name, (M, r, r64) in runs.items():
            _assert_oracle(r, mu_o[:M], s2_o[:M], ymax, "%s %s" % (tag, name))
            _assert_same(r, r64, "%s %s: FP64 flag" % (tag, name))     # small batches take the FP64 kernels whatever the flag
            _assert_oracle(direct[M], mu_o[:M], s2_o[:M], ymax, "%s %s kstar_direct" % (tag, name))
            _assert_close(direct[M], r, "%s %s: kstar_direct vs expansion" % (tag, name))
        _assert_oracle(wide_i8, mu_o, s2_o, ymax, tag + " wide, default path")
        _assert_oracle(wide_fp, mu_o, s2_o, ymax, tag + " wide, FP64")
        _assert_oracle(wide_direct, mu_o, s2_o, ymax, tag + " wide, FP64, kstar_direct")
        _assert_close(wide_direct, wide_fp, tag + " wide: kstar_direct vs expansion")
        if d <= 32:
            # the switches really select other kernels: INT8 vs DMMA, direct differences vs expansion
            assert not np.array_equal(wide_i8[2], wide_fp[2]), tag
            assert not np.array_equal(wide_direct[2], wide_fp[2]), tag
    finally:
        m.close()


@pytest.mark.parametrize("kc", sorted(KERNEL_CLASSES))
@pytest.mark.parametrize("d", GUARD_DIMS)
def test_k1_cancellation_guard_at_high_d(d, kc):
    """short length scales on the unit box: every scaled, centred candidate and training point lies far from the centre, so every
    pair of K1's expansion |x|^2 + |y|^2 - 2 x.y is recomputed from direct differences; with a prior mean (P1 instances, no
    parameter-buffer batch)"""
    from ibo_b200 import _lib
    kind = KERNEL_CLASSES[kc]
    N = 200
    m, o, X, Y, pool = _problem(kind, d, N, 2300, 77 + 1000 * kc + d, scale=0.03, near=0.2, prior=True)
    try:
        # the guard's condition, from the inputs: scaled by 1/theta and centred on the training mean as the model build does
        it = 1.0 / o.kernel.theta
        ctr = (X * it).mean(axis=0)
        yn = np.sum((X * it - ctr) ** 2, axis=1)
        xn = np.sum((pool * it - ctr) ** 2, axis=1)
        assert xn.min() + yn.min() > EXPAND_LIMIT
        ymax = float(Y.max())
        mu_o, s2_o = o.posterior_batch(pool)
        assert s2_o.min() < 0.9 * (1 + NOISE)          # k* is not ~0 everywhere
        tag = "kind %d d %d" % (kind, d)
        lat = _score(m, pool[:100], ymax)
        wide_fp = _score(m, pool, ymax, _lib.FLAG_FP64)
        wide_i8 = _score(m, pool, ymax)
        with options(kstar_direct=1):
            lat_d = _score(m, pool[:100], ymax)
            wide_d = _score(m, pool, ymax, _lib.FLAG_FP64)
        _assert_oracle(lat, mu_o[:100], s2_o[:100], ymax, tag + " latency")
        _assert_oracle(wide_fp, mu_o, s2_o, ymax, tag + " wide FP64")
        _assert_oracle(wide_i8, mu_o, s2_o, ymax, tag + " wide default path")
        _assert_close(lat_d, lat, tag + " latency: kstar_direct")
        _assert_close(wide_d, wide_fp, tag + " wide: kstar_direct")
    finally:
        m.close()


@pytest.mark.parametrize("d", [5, 29])
def test_k1_grid_z_split(d):
    """N = 2049 (17 row-blocks): 1 .. 16 candidate tiles split their n-tiles over grid.z = 16 .. 1 CTAs; FP64 flag, or the mid-size
    rule sends these batches to the INT8 path"""
    from ibo_b200 import _lib
    m, o, X, Y, pool = _problem(orc.K_SE_ARD, d, 2049, 2048, 500 + d)
    try:
        ymax = float(Y.max())
        mu_o, s2_o = o.posterior_batch(pool)
        for M in GRID_Z_BATCHES:
            _assert_oracle(_score(m, pool[:M], ymax, _lib.FLAG_FP64), mu_o[:M], s2_o[:M], ymax, "d %d M %d" % (d, M))
    finally:
        m.close()


# ------------------------------------------------------------------------------------------------------------------------------
# b. K2 latency shapes
# ------------------------------------------------------------------------------------------------------------------------------

# Across shapes the row sums of K2 associate differently, so MT = 4 / 2 / 1 agree with MT = 8 to rounding only.  Largest relative
# differences measured over the eight models below (one B200, 1000 W power limit): mu 1.6e-14 (floor 1e-3), sigma^2 2.9e-14, EI 1.1e-11
# (floor 1e-5: Phi(Z) |mu - ymax| / EI amplifies the posterior's rounding where EI is small).  Bounds: (mu, sigma^2, EI).
K2_MT_SPREAD = (1e-13, 1e-13, 5e-11)


@pytest.mark.parametrize("prior", K2_PRIOR)
@pytest.mark.parametrize("N", K2_NOBS)
def test_k2_latency_shapes(N, prior, plans):
    """trigemm_kernel<1, MT, P1, DEEP> for MT = 8 / 4 / 2 / 1 forced through option narrow_mt, k2_deep = 0 / 1 and pdl = 0 / 1 --
    one model, so narrow_mt changes on a model that has already scored every batch size"""
    from ibo_b200 import _lib
    d = 5
    m, o, X, Y, pool = _problem(orc.K_SE_ARD, d, N, 2048, 300 + N, prior=prior)
    try:
        ymax = float(Y.max())
        mu_o, s2_o = o.posterior_batch(pool)
        # every batch ends at pool index 1096: the same candidate sits at positions 1096, 96, 32, 30 and 0
        slices = {2048: (0, 2048), 97: (1000, 1097), 33: (1064, 1097), 31: (1066, 1097), 1: (1096, 1097)}
        assert sorted(slices) == sorted(K2_BATCHES)
        res = {}
        with options(tiny=0):
            for MT in NARROW_MTS:
                for deep in K2_DEEP:
                    for pdl in (0, 1):
                        with options(narrow_mt=MT, k2_deep=deep, pdl=pdl):
                            for M, (a, b) in slices.items():
                                r = _score(m, pool[a:b], ymax, _lib.FLAG_FP64)
                                _, k2 = plans.take()
                                tag = "N %d prior %s MT %d deep %d pdl %d M %d" % (N, prior, MT, deep, pdl, M)
                                assert [(k["NT"], k["MT"], k["P1"], k["DEEP"], k["PDL"]) for k in k2] == [(1, MT, int(prior), deep, pdl)], \
                                    "%s: recorded %r" % (tag, k2)
                                _assert_oracle(r, mu_o[a:b], s2_o[a:b], ymax, tag)
                                res[(MT, deep, pdl, M)] = r
        spread = [0.0, 0.0, 0.0]
        for MT in NARROW_MTS:
            big = res[(MT, 0, 0, 2048)]
            for M, (a, b) in slices.items():
                ref = res[(MT, 0, 0, M)]
                for deep in K2_DEEP:
                    for pdl in (0, 1):
                        _assert_same(res[(MT, deep, pdl, M)], ref, "N %d MT %d M %d deep %d pdl %d" % (N, MT, M, deep, pdl))
                # same bits wherever the candidate sits and whoever its neighbours are
                for j in range(3):
                    assert np.array_equal(ref[j], big[j][a:b]), "N %d MT %d M %d: position" % (N, MT, M)
            other = res[(8, 0, 0, 2048)]
            spread = [max(spread[0], _rel(big[1], other[1], 1e-3)), max(spread[1], _rel(big[2], other[2], 1e-300)),
                      max(spread[2], _rel(big[0], other[0], EI_FLOOR))]
        plans.note("spread across MT (mu, sigma^2, EI): %.3e %.3e %.3e" % tuple(spread))
        assert all(s <= b for s, b in zip(spread, K2_MT_SPREAD)), spread
    finally:
        m.close()


def test_narrow_mt_takes_effect_on_a_model_that_has_already_scored(plans):
    """option narrow_mt is a run-time switch: a model that has scored a batch of this size under the cost model's plan must run the
    forced shape afterwards, with the bits a fresh model gets under that shape"""
    from ibo_b200 import _lib
    m, o, X, Y, pool = _problem(orc.K_SE_ARD, 4, 640, 33, 11)
    try:
        ymax = float(Y.max())
        first = _score(m, pool, ymax, _lib.FLAG_FP64)
        made, _ = plans.take()
        auto = made[0]["MT"]
        forced = 1 if auto != 1 else 8
        with options(narrow_mt=forced):
            again = _score(m, pool, ymax, _lib.FLAG_FP64)
            _, k2 = plans.take()
            m2 = _lib.Model(orc.K_SE_ARD, list(o.kernel.hyper), X, Y, NOISE)
            try:
                fresh = _score(m2, pool, ymax, _lib.FLAG_FP64)
                plans.take()
            finally:
                m2.close()
        _assert_same(again, fresh, "narrow_mt %d after a scored batch vs a fresh model" % forced)
        assert [k["MT"] for k in k2] == [forced], k2
        back = _score(m, pool, ymax, _lib.FLAG_FP64)
        _, k2 = plans.take()
        assert [k["MT"] for k in k2] == [auto], k2
        _assert_same(back, first, "back to the cost model's plan")
    finally:
        m.close()


def test_k2_latency_shapes_with_a_variance_model(plans):
    """PrefGaussianProcess with observation points: the variance comes from the augmented model's K2 launch (planV) -- both
    models run the forced shape"""
    from ibo_b200 import _lib
    from ibo_b200.gaussianprocess import PrefGaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    rs = np.random.RandomState(21)
    N, d = 300, 4
    X = rs.rand(N, d) * 10
    Y = rs.randn(N)
    A = rs.randn(N, N) * 0.05
    C = np.eye(N) * 5 + A.dot(A.T)
    theta = [5.146, 4.189, 4.622, 5.843]
    gp = PrefGaussianProcess.fromLaplace(GaussianKernel_ard(theta), X, Y, C, noise=0.1)
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, theta, d), X, Y, 0.1, Cinv=np.linalg.inv(C))
    P = rs.rand(5, d) * 10
    gp.addObservationPoint(P)
    augX = np.r_[X, P]
    pad = np.zeros((N + 5, N + 5))
    pad[:N, :N] = np.linalg.inv(C)
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, augX, 0.1) + pad)
    o.augX = augX
    q = rs.rand(200, d) * 10
    q[:60] = augX[rs.randint(N + 5, size=60)] + 0.05 * rs.randn(60, d)
    mu_o, s2_o = o.posterior_batch(q)
    model = gp.model
    plans.take()
    for MT in (8, 2):
        with options(narrow_mt=MT):
            sc, mu, s2, best, bidx = _score(model, q, float(Y.max()), _lib.FLAG_FP64)
        _, k2 = plans.take()
        assert [(k["MT"], k["nb"]) for k in k2] == [(MT, 3), (MT, 3)], k2      # the model's K2, then the variance model's
        assert _rel(mu, mu_o, 1e-3) <= TOL and _rel(s2, s2_o, 1e-300) <= TOL, MT


# ------------------------------------------------------------------------------------------------------------------------------
# c. options that must not change a bit
# ------------------------------------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def wide():
    """N = 2049, d = 6: 17 row-blocks; 20 000 candidates (157 tiles) scored from host buffers (more than 2^17 doubles in and out)"""
    m, o, X, Y, pool = _problem(orc.K_SE_ARD, 6, 2049, 20000, 4242, scale=0.5)
    yield m, X, Y, pool
    m.close()


@pytest.mark.parametrize("M", [20000, 5008])
def test_int8_wide_path_bits_do_not_depend_on_chunking(wide, M):
    """chunk_tiles 1 / 3 / 74 / default x i8_pipe 0 / 1: double-buffered slab and partial planes on two streams, the ragged last
    chunk (5008 = 39 tiles + 16 candidates)"""
    m, X, Y, pool = wide
    ymax = float(Y.max())
    ref = _score(m, pool[:M], ymax)
    for ct in (1, 3, 74, 0):
        for pipe in (0, 1):
            with options(chunk_tiles=ct, i8_pipe=pipe):
                _assert_same(_score(m, pool[:M], ymax), ref, "M %d chunk_tiles %d i8_pipe %d" % (M, ct, pipe))


def test_int8_row_block_groups_do_not_change_bits(wide):
    """i8_rb_per_cta 0 / 1 / 2 / nb (G = 4 / nb / nb/2 / 1 CTAs per candidate tile); 74 tiles (148 64-candidate tiles) keep the
    SM-fill rule from raising G = 1"""
    m, X, Y, pool = wide
    nb = (2049 + 127) // 128
    ymax = float(Y.max())
    ref = _score(m, pool, ymax)
    for per in (0, 1, 2, nb):
        for ct in (74, 0):
            with options(i8_rb_per_cta=per, chunk_tiles=ct):
                _assert_same(_score(m, pool, ymax), ref, "i8_rb_per_cta %d chunk_tiles %d" % (per, ct))


@pytest.mark.parametrize("prior", [False, True])
def test_fp64_wide_path_bits_do_not_depend_on_chunking(prior):
    from ibo_b200 import _lib
    m, o, X, Y, pool = _problem(orc.K_MATERN5_ARD, 7, 2049, 5008, 99, prior=prior)
    try:
        ymax = float(Y.max())
        ref = _score(m, pool, ymax, _lib.FLAG_FP64)
        for ct in (1, 3, 0):
            with options(chunk_tiles=ct):
                _assert_same(_score(m, pool, ymax, _lib.FLAG_FP64), ref, "prior %s chunk_tiles %d" % (prior, ct))
    finally:
        m.close()


def test_latency_shapes_split_into_chunks(plans):
    """chunk_tiles = 1: a 2048-candidate batch in 16 chunks of the latency shapes, PDL across the chunk boundaries; the shape is
    forced (the cost model plans from the chunk's CTA count), and a shape's bits do not depend on the batch"""
    from ibo_b200 import _lib
    m, o, X, Y, pool = _problem(orc.K_SE_ARD, 3, 640, 2048, 5)
    try:
        ymax = float(Y.max())
        for MT in NARROW_MTS:
            with options(narrow_mt=MT, pdl=1):
                ref = _score(m, pool, ymax, _lib.FLAG_FP64)
                with options(chunk_tiles=1):
                    plans.take()
                    got = _score(m, pool, ymax, _lib.FLAG_FP64)
                    _, k2 = plans.take()
            assert [(k["MT"], k["PDL"]) for k in k2] == [(MT, 1)] * 16, k2
            _assert_same(got, ref, "MT %d chunk_tiles 1" % MT)
    finally:
        m.close()


def test_host_buffers_against_resident_candidates(wide):
    """Model.score copies the candidates chunk by chunk two chunks ahead of the kernels through a four-slot event ring; 53 chunks
    make the ring wrap many times"""
    from ibo_b200 import _lib
    m, X, Y, pool = wide
    ymax = float(Y.max())
    M = len(pool)
    assert M * 6 + 3 * M + 2 > 1 << 17             # not staged through the pinned buffer
    rc = _lib.ResidentCandidates(m, pool)
    try:
        for fl in (_lib.FLAG_MODE_CPP, _lib.FLAG_MODE_CPP | _lib.FLAG_FP64):
            ref = m.score(pool, orc.ACQ_EI, ymax, XI, flags=fl)
            for ct in (3, 0):
                tiles = -(-M // 128)
                assert ct == 0 or -(-tiles // ct) >= 10        # chunks of ct 128-candidate tiles
                with options(chunk_tiles=ct):
                    sc, _, _, best, bidx = m.score(pool, orc.ACQ_EI, ymax, XI, flags=fl)
                    out = np.empty(M)
                    rbest, ridx, _ = rc.score(orc.ACQ_EI, ymax, XI, flags=fl, scores_out=out)
                tag = "flags %#x chunk_tiles %d" % (fl, ct)
                assert np.array_equal(sc, ref[0]) and best == ref[3] and bidx == ref[4], tag
                assert np.array_equal(out, sc) and rbest == best and ridx == bidx, tag
    finally:
        rc.close()


def test_int8_guard_pass_across_chunk_boundaries():
    """noise = 1e-6: candidates on / next to training points fall below the INT8 path's sigma^2 guard and are re-scored by the DMMA
    kernels; 16 chunks of 3 tiles must flag, re-score and merge exactly the same candidates as one chunk"""
    from ibo_b200 import _lib
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    N, d, M = 384, 3, 6000
    rs = np.random.RandomState(78)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    gp = GaussianProcess(GaussianKernel_ard([0.08, 0.1, 0.12]), X, Y, noise=1e-6)
    Xs = rs.rand(M, d)
    Xs[10:210] = X[:200]
    Xs[1000:1200] = X[100:300] + 1e-5
    Xs[5999] = X[7]
    fl = _lib.FLAG_MODE_CPP
    ref = gp.model.score(Xs, _lib.ACQ_UCB, Y.max(), 1.5, flags=fl, want_posterior=True)
    ng = gp.model.last_guarded()
    assert ng >= 401
    for ct, pipe in ((3, 1), (3, 0), (1, 1)):
        with options(chunk_tiles=ct, i8_pipe=pipe):
            got = gp.model.score(Xs, _lib.ACQ_UCB, Y.max(), 1.5, flags=fl, want_posterior=True)
        _assert_same(got, ref, "chunk_tiles %d i8_pipe %d" % (ct, pipe))
        assert gp.model.last_guarded() == ng


def test_duplicates_of_the_best_candidate_in_later_chunks(wide):
    """exact copies of the winner further down the batch, in later chunks: the first index wins on both paths"""
    from ibo_b200 import _lib
    m, X, Y, pool = wide
    ymax = float(Y.max())
    for fl in (0, _lib.FLAG_FP64):
        b = _score(m, pool, ymax, fl)[4]
        Xd = pool.copy()
        for j in (40, 7000, 12345, 19999):
            Xd[j] = pool[b]
        first = int(np.flatnonzero((Xd == pool[b]).all(axis=1))[0])
        assert first == min(40, b)
        for ct in (0, 3, 74):
            with options(chunk_tiles=ct):
                sc, mu, s2, best, bidx = _score(m, Xd, ymax, fl)
                tag = "flags %#x chunk_tiles %d" % (fl, ct)
                assert bidx == first and best == sc[first], tag
                assert np.all(sc[[40, 7000, 12345, 19999, b]] == best), tag
