"""smcounter_b200/csrc/smc_py2rand.h -- the CPython-2 hash, dict order, MT19937 seeding and random.sample that the device draw
runs -- compiled with g++ (tests/py2rand_harness.cpp) and compared with smcounter_b200/downsample.py on ~2 000 random sets."""
import ctypes as C
import math
import os
import random
import shutil
import subprocess

import numpy as np
import pytest

from py2_sets import SIZES_LARGE, code_hash, hashes_of, make_sets, reference_draw
from smcounter_b200.downsample import py2_dict_key_order, py2_string_hash

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    so = str(tmp_path_factory.mktemp("py2rand") / "libpy2rand.so")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC",
                        "-I", os.path.join(HERE, "..", "smcounter_b200", "csrc"), "-o", so, os.path.join(HERE, "py2rand_harness.cpp")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    h = C.CDLL(so)
    h.h_hash_umi2.argtypes, h.h_hash_umi2.restype = [C.c_uint64], C.c_int64
    h.h_hash_decimal.argtypes, h.h_hash_decimal.restype = [C.c_int64], C.c_int64
    h.h_setsizes.argtypes, h.h_setsizes.restype = [C.c_int64, C.c_void_p], None
    h.h_dict_order.argtypes, h.h_dict_order.restype = [C.c_void_p, C.c_int64, C.c_void_p], None
    h.h_random.argtypes, h.h_random.restype = [C.c_int64, C.c_int64, C.c_void_p], None
    h.h_draw.argtypes, h.h_draw.restype = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p], None
    return h


@pytest.fixture(scope="module")
def sets():
    return make_sets()


def test_setsize_is_the_integer_form_of_the_log_formula(lib):
    kmax = 1_000_000
    got = np.zeros(kmax + 1, np.int64)
    lib.h_setsizes(kmax, got.ctypes.data)
    want = np.array([21 + (4 ** int(math.ceil(math.log(k * 3, 4))) if k > 5 else 0) for k in range(kmax + 1)], dtype=np.int64)
    assert np.array_equal(got, want)


def test_string_hashes(lib, sets):
    codes = {c for s in sets[0] for c in s[0] if not c >> 63} | {1}
    for c in codes:
        assert lib.h_hash_umi2(c) == code_hash(c, None), hex(c)
    for v in list(range(0, 2000)) + [random.Random(3).randrange(1, 1 << 40) for _ in range(2000)]:
        assert lib.h_hash_decimal(v) == py2_string_hash(str(v)), v


def test_seeding(lib, sets):
    for _, _, pos1, _ in sets[0]:
        got = np.zeros(8, np.float64)
        lib.h_random(pos1, 8, got.ctypes.data)
        rng = random.Random()
        rng.seed(py2_string_hash(str(pos1)) & ((1 << 64) - 1))
        assert got.tolist() == [rng.random() for _ in range(8)], pos1


def test_dict_order_and_draw_equal_downsample_py(lib, sets):
    branches = set()
    ks = set()
    for codes, strs, pos1, k in sets[0]:
        n = len(strs)
        h = hashes_of(strs)
        order = np.zeros(max(n, 1), np.uint32)
        lib.h_dict_order(h.ctypes.data, n, order.ctypes.data)
        index = {s: i for i, s in enumerate(strs)}
        assert order[:n].tolist() == [index[s] for s in py2_dict_key_order(strs)], n
        out = np.zeros(max(k, 1), np.uint32)
        lib.h_draw(h.ctypes.data, n, pos1, k, out.ctypes.data)
        assert out[:k].tolist() == reference_draw(strs, pos1, k), (n, k, pos1)
        setsize = 21 + (4 ** int(math.ceil(math.log(k * 3, 4))) if k > 5 else 0)
        branches.add("pool" if n <= setsize else "selection")
        ks.add("edge" if k in (0, 1, 5, 6, n - 1, n) else "random")
    assert branches == {"pool", "selection"} and ks == {"edge", "random"}
    sizes = [len(s[1]) for s in sets[0]]
    assert len(sizes) >= 2000 and min(sizes) == 1 and max(sizes) == max(SIZES_LARGE)
    lens = {len(s) for st in sets[0] for s in st[1]}
    assert 0 in lens and 31 in lens and any(c >> 63 for st in sets[0] for c in st[0])


def test_device_draw_constants_mirror_the_header():
    import re
    from smcounter_b200 import _ffi
    hdr = open(os.path.join(HERE, "..", "include", "smc_b200.h")).read()
    for cname, val in (("SMC_DS_FLAG", _ffi.DS_FLAG), ("SMC_DS_DEVICE", _ffi.DS_DEVICE), ("SMC_ST_DOWNSAMPLED", _ffi.ST_DOWNSAMPLED)):
        assert int(re.search(r"#define\s+%s\s+(\d+)" % cname, hdr).group(1)) == val, cname
