"""The number formatting of the device score-file writer (csrc/blp_json_format.cuh), compiled for
the host with nvcc into a throwaway shared object and compared byte for byte with what json.dumps
writes: float.__repr__ for finite doubles, NaN / Infinity / -Infinity, int.__repr__ for ints.
No GPU needed; the library itself has no CPU path -- this object exists only inside the test."""
import ctypes
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

CSRC = os.path.join(ROOT, 'bipartite-link-prediction_b200', 'csrc')

SHIM = r'''
#include "blp_json_format.cuh"
static const blp_json::Pow5Tables kTables = {&blp_pow5_inv_split[0][0], &blp_pow5_split[0][0]};
// every value followed by '\n'; returns the bytes written
extern "C" long long fmt_doubles(const double* v, long long n, char* out) {
    long long at = 0;
    for (long long i = 0; i < n; ++i) {
        at += blp_json::format_double(v[i], out + at, kTables);
        out[at++] = '\n';
    }
    return at;
}
extern "C" long long fmt_ints(const long long* v, long long n, char* out) {
    long long at = 0;
    for (long long i = 0; i < n; ++i) {
        at += blp_json::format_int64(v[i], out + at);
        out[at++] = '\n';
    }
    return at;
}
'''


@pytest.fixture(scope='module')
def fmt(tmp_path_factory):
    d = tmp_path_factory.mktemp('json_format')
    src, so = str(d / 'shim.cu'), str(d / 'shim.so')
    with open(src, 'w') as fh:
        fh.write(SHIM)
    nvcc = os.environ.get('NVCC', 'nvcc')
    res = subprocess.run([nvcc, '-O2', '-std=c++17', '-Xcompiler', '-fPIC', '-shared', '-I', CSRC,
                          src, '-o', so], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 0, res.stdout
    lib = ctypes.CDLL(so)
    for f in (lib.fmt_doubles, lib.fmt_ints):
        f.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p]
        f.restype = ctypes.c_longlong
    return lib


def _run(fn, arr, width):
    out = np.empty(arr.size * (width + 1) + 1, dtype=np.uint8)
    n = fn(arr.ctypes.data, arr.size, out.ctypes.data)
    return out[:n].tobytes().decode('ascii')


def check_doubles(fmt, values):
    arr = np.ascontiguousarray(values, dtype=np.float64)
    got = _run(fmt.fmt_doubles, arr, 24)
    want = ''.join(json.dumps(x) + '\n' for x in arr.tolist())
    if got != want:
        g, w = got.split('\n'), want.split('\n')
        bad = [i for i in range(len(w)) if g[i] != w[i]]
        pytest.fail('%d of %d doubles differ, first: %r -> %r (want %r)'
                    % (len(bad), arr.size, arr[bad[0]], g[bad[0]], w[bad[0]]))


def with_neighbours(x):
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(over='ignore'):
        return np.concatenate([np.nextafter(x, -np.inf), x, np.nextafter(x, np.inf)])


def test_jaccard_ratios(fmt):
    """Every cn/uni with 1 <= cn <= uni <= 2000 (the jaccard column's values)."""
    uni = np.concatenate([np.full(u, u) for u in range(1, 2001)]).astype(np.float64)
    cn = np.concatenate([np.arange(1, u + 1) for u in range(1, 2001)]).astype(np.float64)
    check_doubles(fmt, cn / uni)


def test_random_bit_patterns(fmt):
    bits = np.random.default_rng(20181).integers(0, 2 ** 64, size=1_200_000, dtype=np.uint64)
    v = bits.view(np.float64)
    v = v[np.isfinite(v)]
    assert v.size >= 1_000_000
    check_doubles(fmt, v)


def test_powers_of_two(fmt):
    check_doubles(fmt, [math.ldexp(1.0, e) for e in range(-1074, 1024)])


def test_decimal_powers_and_neighbours(fmt):
    p = np.array([float('1e%d' % k) for k in range(-323, 309)])
    check_doubles(fmt, with_neighbours(p))
    check_doubles(fmt, -with_neighbours(p))


def test_notation_switch_and_special_values(fmt):
    tiny = sys.float_info.min                      # smallest normal
    vals = [1e-4, 1e-5, 9.999999999999999e-05, 0.00011, 1e16, 9999999999999998.0, 1e15,
            123456789012345680.0, 1.5e16, 0.1, 0.2, 0.3, 1 / 3, 2 / 3, 100.0, 1e22, 1e23, 5e-324,
            tiny, tiny - 5e-324, sys.float_info.max, 2.0 ** 53, 2.0 ** 53 + 2, 2.0 ** 53 - 1,
            2.0 ** 54, 0.0, 1.0, 9007199254740993.0, 4.35, 2.5, 0.5, 1.7976931348623157e308]
    check_doubles(fmt, with_neighbours(vals))
    check_doubles(fmt, -with_neighbours(vals))
    check_doubles(fmt, [-0.0, 0.0, float('nan'), float('inf'), float('-inf')])
    # the smallest subnormals, and the subnormal / normal boundary with a run of ulps either side
    check_doubles(fmt, np.arange(0, 65, dtype=np.int64).view(np.float64))
    check_doubles(fmt, (np.int64(np.float64(tiny).view(np.int64)) +
                        np.arange(-200, 201, dtype=np.int64)).view(np.float64))


def test_adamic_adar_fixed_point_values(fmt):
    """adamic is a Q1.31 fixed-point sum converted to double: k / 2^31."""
    k = np.concatenate([np.arange(0, 1 << 20, dtype=np.int64),
                        np.random.default_rng(7).integers(0, 1 << 45, size=300_000)])
    check_doubles(fmt, k.astype(np.float64) / 2.0 ** 31)


def test_ints_format_like_int_repr(fmt):
    ext = [0, 1, -1, 9, 10, -10, 2 ** 31 - 1, -2 ** 31, 2 ** 32, 2 ** 63 - 1, -2 ** 63,
           10 ** 18, -10 ** 18, 10 ** 18 - 1, 999999999999999999]
    rnd = np.random.default_rng(3).integers(-2 ** 63, 2 ** 63 - 1, size=200_000, dtype=np.int64)
    small = np.arange(-1000, 1001, dtype=np.int64)
    arr = np.concatenate([np.array(ext, dtype=np.int64), rnd, small,
                          10 ** np.arange(19, dtype=np.int64), -10 ** np.arange(19, dtype=np.int64)])
    got = _run(fmt.fmt_ints, arr, 20)
    assert got == ''.join(repr(int(x)) + '\n' for x in arr.tolist())


def test_pow5_table_is_what_the_generator_computes():
    """csrc/blp_json_pow5.h is generated by tools/gen_json_pow5.py; regenerate and compare."""
    gen = os.path.join(ROOT, 'tools', 'gen_json_pow5.py')
    res = subprocess.run([sys.executable, gen, '--stdout'], stdout=subprocess.PIPE, check=True)
    with open(os.path.join(CSRC, 'blp_json_pow5.h'), 'rb') as fh:
        assert fh.read() == res.stdout
