"""Which kernels score a batch is decided once, by plan_score (ibo_b200/csrc/score.cu), for every scoring entry point.  Two corners
of that decision:

- a batch above option narrow_max whose candidates fit K1's parameter buffer, on a model that takes the INT8 path: the INT8 K1
  reads its candidates from device memory, so the batch must be copied there;
- flag bits the C ABI does not document (29 and 30 among them) change nothing: the same kernels run and give the same bits."""
import numpy as np
import pytest

from oracle import ibo_oracle as orc
from test_gpu_dispatch import _assert_same, _problem, _score, options, plans  # noqa: F401  (plans: fixture)

pytestmark = pytest.mark.gpu

PRIVATE_BITS = [1 << 29, 1 << 30, (1 << 29) | (1 << 30)]


def test_int8_batch_above_narrow_max_that_fits_the_parameter_buffer(plans):
    """N = 2048, d = 2 (16 row-blocks), narrow_max = 64: 100-point batches (200 doubles, within the parameter buffer) take the INT8
    path and give the bits of the same rows of one 70 000-candidate INT8 call"""
    m, o, X, Y, pool = _problem(orc.K_SE_ARD, 2, 2048, 70000, 2048)
    try:
        ymax = float(Y.max())
        with options(narrow_max=64):
            big = _score(m, pool, ymax)
            for a in (0, 4321, 35000, 69900):
                got = _score(m, pool[a:a + 100], ymax)
                made, k2 = plans.take()
                assert made == [] and k2 == [], "offset %d: FP64 plans %r, K2 launches %r" % (a, made, k2)     # the INT8 kernels
                for j, what in enumerate(("scores", "mu", "sigma^2")):
                    assert np.array_equal(got[j], big[j][a:a + 100]), "offset %d: %s" % (a, what)
    finally:
        m.close()


@pytest.mark.parametrize("N, M", [(640, 33), (100, 50), (100, 300), (640, 3000)])
def test_undocumented_flag_bits_change_nothing(N, M, plans):
    """N = 640 (a latency plan), one row-block (the fused kernel: no K2 line; 50 points in the parameter buffer, 300 from mapped
    memory) and a 3000-point batch (INT8 path, and the FP64 throughput shape with FLAG_FP64)"""
    from ibo_b200 import _lib
    m, o, X, Y, pool = _problem(orc.K_SE_ARD, 3, N, M, 7 + N + M)
    try:
        ymax = float(Y.max())
        for fl in (0, _lib.FLAG_FP64):
            _score(m, pool, ymax, fl)                  # a latency plan is printed when it is made: make it before recording
            plans.take()
            ref = _score(m, pool, ymax, fl)
            ref_plans = plans.take()
            ref_post = m.posterior(pool, flags=_lib.FLAG_MODE_PY | fl)
            post_plans = plans.take()
            if N <= 128:
                assert ref_plans[1] == [] and post_plans[1] == [], (ref_plans, post_plans)
            for bits in PRIVATE_BITS:
                tag = "N %d M %d flags %#x" % (N, M, fl | bits)
                got = _score(m, pool, ymax, fl | bits)
                assert plans.take() == ref_plans, tag
                _assert_same(got, ref, tag)
                post = m.posterior(pool, flags=_lib.FLAG_MODE_PY | fl | bits)
                assert plans.take() == post_plans, tag + ": posterior"
                assert np.array_equal(post[0], ref_post[0]) and np.array_equal(post[1], ref_post[1]), tag + ": posterior"
    finally:
        m.close()
