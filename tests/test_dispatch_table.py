"""CPU check that tests/test_gpu_dispatch.py reaches every template instance of the scoring path's dispatch, parsed from the sources
(ibo_b200/csrc/score.cu, score_i8.cuh): the FP64 K1 arms kstar_mma_kernel<DP4, KC> (and the switch's default arm), the INT8 K1 buckets
kstar_i8_kernel<KC, DMAX>, and the K2 latency shapes trigemm_kernel<1, MT, ...>.  Adding a bucket that no GPU case reaches fails here."""
import os
import re

import test_gpu_dispatch as gd

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ibo_b200", "csrc")


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _body(txt, start):
    """text of the C++ function whose definition starts at `start`, up to its closing brace at column 0"""
    i = txt.index(start)
    return txt[i:txt.index("\n}\n", i)]


def test_fp64_k1_arms_are_covered():
    txt = _src("score.cu")
    sw = _body(txt, "static void launch_kstar(")
    arms = re.findall(r"case (\d+): launch_kstar_mma<(\d+)>", sw)
    assert arms and all(a == b for a, b in arms)
    default = int(re.search(r"default: launch_kstar_mma<(\d+)>", sw).group(1))
    # the expansion runs while ceil(d / 4) <= limit, the direct-difference kernel beyond
    limit = int(re.search(r"\(m->d \+ 3\) / 4 <= (\d+)", txt).group(1))
    instances = {int(a) for a, _ in arms} | {default}
    assert instances == set(range(1, limit + 1))
    reached = set()
    for d in gd.DIMS:
        dp4 = (d + 3) // 4
        if dp4 <= limit:
            reached.add(dp4 if dp4 in {int(a) for a, _ in arms} else default)
    assert reached == instances, sorted(instances - reached)
    assert default in reached                                     # the switch's default arm
    assert any((d + 3) // 4 > limit for d in gd.DIMS)             # and the direct-difference kernel
    classes = {int(c) for c in re.findall(r"kstar_mma_kernel<DP4, (\d+)><<<", _body(txt, "static void launch_kstar_mma("))}
    assert classes == set(gd.KERNEL_CLASSES) == {0, 1, 2}
    # K1's parameter-buffer batch: both sides of the boundary at every d
    assert gd.CAND_INLINE == int(re.search(r"constexpr int CAND_INLINE = (\d+);", _src("common.cuh")).group(1))


def test_int8_k1_buckets_are_covered():
    txt = _src("score_i8.cuh")
    sw = _body(txt, "static void launch_kstar_i8(")
    bounded = [(int(a), int(b)) for a, b in re.findall(r"if \(d <= (\d+)\) launch_kstar_i8_d<(\d+)>", sw)]
    assert bounded and all(a == b for a, b in bounded)
    last = int(re.search(r"else launch_kstar_i8_d<(\d+)>", sw).group(1))
    dmax_eligible = int(re.search(r"m->d > (\d+) \|\|", _src("score.cu")).group(1))     # i8_eligible: d above it -> FP64
    assert last == dmax_eligible
    buckets = [b for _, b in bounded] + [last]
    reached = set()
    for d in gd.DIMS:
        if d <= dmax_eligible:
            reached.add(next(b for b in buckets if d <= b))
    assert reached == set(buckets), sorted(set(buckets) - reached)
    classes = {int(c) for c in re.findall(r"kstar_i8_kernel<(\d+), DMAX><<<", _body(txt, "static void launch_kstar_i8_d("))}
    assert classes == set(gd.KERNEL_CLASSES)


def test_k2_latency_shapes_are_covered():
    txt = _src("score.cu")
    sw = _body(txt, "static int launch_trigemm(")
    arms = [(int(a), int(b)) for a, b in re.findall(r"pl\.MT == (\d+)\) launch_k2_shape<1, (\d+)>", sw)]
    assert arms and all(a == b for a, b in arms)
    shapes = {b for _, b in arms} | {int(re.search(r"else launch_k2_shape<1, (\d+)>", sw).group(1))}
    mts = {int(v) for v in re.search(r"const int mts\[\d+\] = \{([0-9, ]+)\};", txt).group(1).split(",")}
    attrs = {int(v) for v in re.findall(r"set_k2_attr<1, (\d+)>\(\)", txt)}
    assert shapes == mts == attrs == set(gd.NARROW_MTS)
    # both template flags of every shape: P1 (prior mean) and DEEP (option k2_deep 0 / 1)
    assert set(gd.K2_PRIOR) == {False, True} and set(gd.K2_DEEP) == {0, 1}
    # models whose last row-block holds one live row, and one with a single row-block
    assert any(n % 128 == 1 for n in gd.K2_NOBS) and any(n <= 128 for n in gd.K2_NOBS)
    assert gd.GRID_Z_BATCHES == [100, 200, 450, 1000, 2048]
