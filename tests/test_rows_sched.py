"""The slot windows of the row-owned variant of kernel 2 (indelope_b200/csrc/ksw2_rows_sched.cuh), built here as plain C++
(tests/native/rows_sched_host.cpp) and checked against the per-thread, per-diagonal rule they replace -- no GPU needed.  On the GPU the
same windows steer ksw2_rows, whose results tests/test_gpu_ksw2.py compares with the reference bit for bit."""
import ctypes as C
import os
import random
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NOUT = 6


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    src = os.path.join(HERE, "native", "rows_sched_host.cpp")
    so = str(tmp_path_factory.mktemp("rows_sched") / "librows_sched_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-x", "c++", "-I", os.path.join(ROOT, "indelope_b200", "csrc"), src, "-o", so])
    lib = C.CDLL(so)
    I4 = C.c_int * 4
    lib.idl_test_rows_warp.argtypes = [I4, I4, I4, C.POINTER(C.c_longlong)]
    lib.idl_test_rows_shapes.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_longlong)]
    return lib


def _check(out):
    assert out[0] == 0, "a thread has a lane inside the target outside the warp's live window"
    assert out[1] == 0, "the interior window holds a thread whose word is not wholly inside the target"
    assert out[2] == 0, "ksw_rows_lane_on differs from the per-diagonal rule"


def test_every_shape(L):
    """qlen 1..160 (every read the variant serves) against tlen 1..600: four equal groups, and one group beside three without an alignment"""
    out = (C.c_longlong * NOUT)()
    L.idl_test_rows_shapes(160, 600, out)
    _check(out)
    assert out[3] > 0 and out[4] > out[3] and out[5] > 0


def test_mixed_warps(L):
    """four groups of different shapes in one warp, some of them without a live alignment (no task, or an empty query or target)"""
    rng = random.Random(11)
    I4 = C.c_int * 4
    total = (C.c_longlong * NOUT)()
    for k in range(4000):
        valid, ql, tl = [], [], []
        for g in range(4):
            dead = rng.random() < 0.15
            valid.append(0 if dead and rng.random() < 0.5 else 1)
            q = rng.randint(1, 160) if k % 2 else rng.randint(120, 160)   # half of the warps alike, as the length-sorted tasks are
            t = rng.randint(1, 600) if k % 3 else rng.randint(100, 400)
            if dead and valid[-1]:
                q, t = (0, t) if rng.random() < 0.5 else (q, 0)
            ql.append(q); tl.append(t)
        out = (C.c_longlong * NOUT)()
        L.idl_test_rows_warp(I4(*valid), I4(*ql), I4(*tl), out)
        _check(out)
        for i in range(NOUT):
            total[i] += out[i]
    assert total[3] > 0 and total[5] > 0


def test_warp_with_a_dead_group_has_no_interior(L):
    """a group without a live alignment empties the interior window: its threads never run a word"""
    I4 = C.c_int * 4
    for valid, ql, tl in (([1, 1, 1, 0], [150, 150, 150, 150], [233, 233, 233, 233]),
                          ([1, 1, 1, 1], [150, 0, 150, 150], [233, 233, 233, 233]),
                          ([1, 1, 1, 1], [150, 150, 150, 150], [233, 0, 233, 233])):
        out = (C.c_longlong * NOUT)()
        L.idl_test_rows_warp(I4(*valid), I4(*ql), I4(*tl), out)
        _check(out)
        assert out[3] == 0 and out[4] > 0
