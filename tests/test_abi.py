"""CPU tests of the drop-in boundary: the C-ABI library loads without a GPU, exports every symbol
include/ibo_b200.h declares, and its compute entry points fail loudly (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest

from ibo_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "ibo_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    names = set(re.findall(r"\b(ibo_[a-z_0-9]+|direct|acqmaxGP)\s*\(", txt))
    names -= {"ibo_batch_objective_t"}
    return names


def test_library_exports_every_declared_symbol():
    L = _lib.lib()
    declared = header_symbols()
    assert declared == set(_lib.EXPORTED), (declared ^ set(_lib.EXPORTED))
    for name in declared:
        assert hasattr(L, name), "missing export %s" % name


def test_version_and_error_strings():
    L = _lib.lib()
    assert b"sm_100a" in L.ibo_version()
    assert isinstance(L.ibo_last_error(), bytes)


def test_bad_arguments_are_rejected_without_touching_a_gpu():
    L = _lib.lib()
    h = ctypes.c_void_p()
    info = ctypes.c_int(0)
    x = np.zeros((2, 2)); y = np.zeros(2); hy = np.ones(2)
    rc = L.ibo_model_create(0, 99, _lib.dptr(hy), 2, _lib.dptr(x), _lib.dptr(y), 2, 2, 0.1, None,
                            0, _lib.dptr(y), _lib.dptr(y), 0.0, _lib.dptr(y), _lib.dptr(y), ctypes.byref(h), ctypes.byref(info))
    assert rc == _lib.E_BADARG
    assert L.ibo_posterior_batch(None, _lib.dptr(x), 2, 0, None, None) == _lib.E_BADARG


@pytest.mark.skipif(_lib.lib().ibo_device_count() > 0, reason="a GPU is present")
def test_no_cpu_fallback():
    """Without a device every product entry point must fail loudly instead of computing on the CPU."""
    rs = np.random.RandomState(0)
    X = rs.rand(8, 2); Y = rs.rand(8)
    with pytest.raises(_lib.IBOError) as ei:
        _lib.Model(_lib.KERNEL_SE_ISO, [0.3], X, Y, 0.1)
    assert ei.value.code == _lib.E_CUDA
    with pytest.raises(_lib.IBOError):
        _lib.require_gpu()
    # legacy symbol: NULL on failure (reference convention, cpp/optimizeGP.cpp:342-346)
    L = _lib.lib()
    lb = np.zeros(2); ub = np.ones(2); invR = np.eye(8); hy = np.array([0.3]); z = np.zeros(1)
    res = L.acqmaxGP(2, _lib.dptr(lb), _lib.dptr(ub), _lib.dptr(invR), _lib.dptr(X), _lib.dptr(Y), 8, 0, 1, _lib.dptr(hy),
                     0, _lib.dptr(z), _lib.dptr(z), 0.0, _lib.dptr(z), _lib.dptr(z), 0.01, 0.1, 5, 30, 100)
    assert not res


def documented_options():
    """name -> default from the "options" section of the header ("name (default)" entries)"""
    txt = open(os.path.join(ROOT, "include", "ibo_b200.h")).read()
    sec = txt[txt.index("---- options"):txt.index("int ibo_set_option")]
    return {n: int(v) for n, v in re.findall(r"\b([a-z][a-z0-9_]+) \((-?\d+)\)", sec)}


def test_options_are_exactly_what_the_header_says():
    """the header documents exactly the library's options, each exists with the documented default (read in a fresh process: other
    tests change options), unknown and removed names are rejected, values round-trip, and IBO_<NAME> presets an option when the
    library is loaded"""
    import subprocess
    import sys
    opts = documented_options()
    assert set(opts) == {"int8", "i8_min_batch", "i8_guard", "i8_pipe", "i8_rb_per_cta", "chunk_tiles", "narrow_max", "narrow_mt",
                         "k2_deep", "pdl", "kstar_direct", "tiny", "debug_plan", "direct_timing", "shard_min", "tiny_server", "chol_pair"}
    assert opts["int8"] == 1 and opts["i8_min_batch"] == -1 and opts["tiny_server"] == 1
    code = ("import sys; sys.path.insert(0, %r)\nfrom ibo_b200 import _lib\n"
            "print(' '.join('%%s=%%d' %% (n, _lib.get_option(n)) for n in %r))" % (ROOT, sorted(opts)))
    env = {k: v for k, v in os.environ.items() if not k.startswith("IBO_")}
    out = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, text=True, check=True).stdout.split()
    assert dict((kv.split("=")[0], int(kv.split("=")[1])) for kv in out) == opts
    env["IBO_INT8"] = "0"; env["IBO_CHOL_PAIR"] = "1"
    out = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, text=True, check=True).stdout.split()
    got = dict((kv.split("=")[0], int(kv.split("=")[1])) for kv in out)
    assert got["int8"] == 0 and got["chol_pair"] == 1 and got["i8_guard"] == 1
    L = _lib.lib()
    v = ctypes.c_long(0)
    for name in (b"no_such_option", b"i8_ntm", b"i8_dbg"):
        assert L.ibo_set_option(name, 1) == _lib.E_BADARG and L.ibo_get_option(name, ctypes.byref(v)) == _lib.E_BADARG
    old = _lib.get_option("narrow_mt")
    try:
        _lib.set_option("narrow_mt", 4)
        assert _lib.get_option("narrow_mt") == 4
    finally:
        _lib.set_option("narrow_mt", old)
