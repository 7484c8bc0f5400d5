"""CPU check of the MMA schedule of trigemm_i8_kernel (ibo_b200/csrc/score_i8.cuh), parsed from the source: every k-step issues
A_t x [B_u0 .. B_u0+n-1] instructions whose 64-column output blocks land on TMEM columns 64 (t + u - 2).  Emulated on an accumulator
array pre-filled with garbage, the schedule must leave exactly D_g = sum_k sum_{t+u=g} A_t B_u^T in every group -- in particular the
first k-step must overwrite every group exactly once before anything accumulates into it -- and must stay within the 448 accumulator
columns."""
import os
import re

import numpy as np

SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ibo_b200", "csrc", "score_i8.cuh")


def schedule():
    txt = open(SRC).read()
    body = txt[txt.index("#define I8_MMA(t, u0, n, acc)"):txt.index("#undef I8_MMA\n")]
    pat = re.compile(r"I8_MMA\((\d+), (\d+), (\d+), (first|1u)\)")
    return [(int(a), int(b), int(c), d == "first") for a, b, c, d in pat.findall(body)]


def test_mma_schedule_builds_the_group_sums():
    S, gmax = 7, 8
    ops = schedule()
    assert sum(n for _, _, n, _ in ops) == sum(1 for t in range(1, S + 1) for u in range(1, S + 1) if t + u <= gmax) == 28
    assert len(ops) == 10
    rs = np.random.RandomState(0)
    ksteps, M, NC, K = 3, 16, 8, 32                 # 8 "candidates" per 64-column block stand-in
    A = rs.randint(-64, 64, size=(ksteps, S, M, K)).astype(np.int64)
    B = rs.randint(-128, 128, size=(ksteps, S, NC, K)).astype(np.int64)
    tmem = rs.randint(-10 ** 6, 10 ** 6, size=(M, 7 * NC)).astype(np.int64)      # garbage left by the previous row-block
    for j in range(ksteps):
        for t, u0, n, first in ops:
            assert 1 <= t <= S and u0 >= 1 and u0 + n - 1 <= S and t + u0 + n - 1 <= gmax
            assert n * 64 in (64, 128, 192, 256)                                   # legal UMMA N for M = 128
            col = (t + u0 - 2) * NC
            assert col + n * NC <= 7 * NC                                          # 448 accumulator columns
            prod = np.concatenate([A[j, t - 1] @ B[j, u - 1].T for u in range(u0, u0 + n)], axis=1)
            if first and j == 0:
                tmem[:, col:col + n * NC] = prod
            else:
                tmem[:, col:col + n * NC] += prod
    for g in range(2, gmax + 1):
        want = sum(A[j, t - 1] @ B[j, g - t - 1].T for j in range(ksteps) for t in range(1, S + 1) if 1 <= g - t <= S)
        assert np.array_equal(tmem[:, (g - 2) * NC:(g - 1) * NC], want), g
