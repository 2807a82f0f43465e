"""CPU test of odam_b200/csrc/sq_math.cuh (the same source the kernels compile): accuracy against x87 extended
precision, and that rounding to float gives the correctly rounded result on the sampler's domain."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def m(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("sq_math") / "libsq_math_host_test.so")
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-std=c++17", "-o", so,
                    os.path.join(REPO, "odam_b200", "csrc", "sq_math_host.cpp"), "-lm"], check=True)
    return C.CDLL(so)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_sincos(m):
    rng = np.random.default_rng(0)
    n = 400_000
    th = rng.uniform(-np.pi, np.pi, n).astype(np.float32)
    pi = np.float32(np.pi)
    th[:8] = [0, pi, -pi, pi / 2, -pi / 2, 1e-6, pi / 4, 3 * pi / 4]
    s, c = np.zeros(n), np.zeros(n)
    m.sq_math_sincos(_p(th), n, _p(s), _p(c))
    tl = th.astype(np.longdouble)
    sr, cr = np.sin(tl), np.cos(tl)
    assert np.max(np.abs(s - sr) / np.abs(sr).clip(1e-300)) < 1e-15
    assert np.max(np.abs(c - cr) / np.abs(cr).clip(1e-300)) < 1e-15
    assert np.array_equal(s.astype(np.float32), sr.astype(np.float32))
    assert np.array_equal(c.astype(np.float32), cr.astype(np.float32))
    assert np.float32(c[3]) < 0 and np.float32(s[1]) < 0   # cosf(fl(pi/2)), sinf(fl(pi)): the H3 signs


def test_pow01(m):
    rng = np.random.default_rng(1)
    n = 400_000
    x = np.concatenate([rng.uniform(0, 1, n // 2), 10 ** rng.uniform(-8, 0, n // 2)]).astype(np.float32)
    x[:5] = [1.0, 4.371139e-08, 8.742278e-08, 1e-6, 0.0]
    p = rng.uniform(0.2, 1.6, n).astype(np.float32)
    p[:50] = 0.2
    out = np.zeros(n)
    m.sq_math_pow01(_p(x), _p(p), n, _p(out))
    ref = np.power(x.astype(np.longdouble), p.astype(np.longdouble))
    nz = x > 0
    assert np.max(np.abs(out[nz] - ref[nz]) / ref[nz]) < 2e-14
    assert np.array_equal(out.astype(np.float32), ref.astype(np.float32))
    assert out[0] == 1.0 and out[4] == 0.0


def test_glibc_faithful_cosf_sinf_powf_bit_identical_to_libm(m):
    """The sampler's transcendentals are libm's algorithms restated (sq_glibc_*): on an x86-64 host whose libm takes
    the FMA ifunc variants (any AVX2+FMA CPU, glibc >= 2.28) the restatement must agree with libm bit for bit on the
    sampler's domain.  Skipped where libm resolves to the non-FMA variants (different roundings by design)."""
    import ctypes.util
    flags = open("/proc/cpuinfo").read()
    if " fma" not in flags or " avx2" not in flags:
        pytest.skip("host libm uses the non-FMA variants")
    M = C.CDLL(ctypes.util.find_library("m"))
    for f in (M.cosf, M.sinf, M.powf):
        f.restype = C.c_float
    M.cosf.argtypes = M.sinf.argtypes = [C.c_float]
    M.powf.argtypes = [C.c_float, C.c_float]
    rng = np.random.default_rng(3)
    n = 120_000
    x = rng.uniform(-3.2, 3.2, n).astype(np.float32)
    pi = np.float32(np.pi)
    x[:10] = [0, pi, -pi, pi / 2, -pi / 2, 1e-6, pi / 4, 3 * pi / 4, 0.75, -0.7499]
    x[10:4000] = (10 ** rng.uniform(-9, 0, 3990)).astype(np.float32)
    p = rng.uniform(0.2, 1.6, n).astype(np.float32)
    p[:100] = 0.2
    c, s, pw = (np.zeros(n, np.float32) for _ in range(3))
    m.sq_math_glibc(_p(x), _p(p), n, _p(c), _p(s), _p(pw))
    rc = np.array([M.cosf(float(v)) for v in x], np.float32)
    rs = np.array([M.sinf(float(v)) for v in x], np.float32)
    rp = np.array([M.powf(float(abs(v)), float(q)) for v, q in zip(x, p)], np.float32)
    assert np.array_equal(c, rc) and np.array_equal(s, rs) and np.array_equal(pw, rp)
    assert c[3] < 0 and s[1] < 0   # cosf(fl(pi/2)), sinf(fl(pi)): the H3 signs
