"""GPU twin of tests/test_power_helpers.py: the same instances, operands, policies and contract,
compiled for sm_100a with the hardware reciprocal seed (MUFU.RCP64H) in the half powers; and the
per-point pow of flavour "glibc-all" (inflx_gl_pow_m) against the host libm's bits at the same
operands."""
import os

import numpy as np
import pytest

from test_power_helpers import (HARD, KINDS, N_RANGE, NATIVE, arguments, build_host_checker,
                                check_instance, exponent, reference, same_bits)

pytestmark = pytest.mark.gpu

# x^(N+1/2): the correction d of sqrt(x) = s + d is scaled by the ~2^-23 seed reciprocal, which
# leaves the double-double value ~2^-76 (relative, ~2^-23 ulp) from the power
HARD_SEEDED = 2.0**-20


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    return build_host_checker(tmp_path_factory.mktemp("pow"))


@pytest.fixture(scope="module")
def device():
    from gpu_kernels import Module

    with open(os.path.join(NATIVE, "pow_check.cpp")) as fh:
        return Module("#define INFLX_POW_CHECK_DEVICE 1\n" + fh.read())


@pytest.mark.parametrize("kind", sorted(KINDS))
def test_power_helper_on_the_device_is_correctly_rounded(host, device, kind):
    hard = HARD if kind < 2 else HARD_SEEDED
    off = total = 0
    for n in N_RANGE[kind]:
        x = arguments(kind, n)
        m = x.size
        cr, dist, _ = reference(host, kind, n, x)
        exact, spec, flag = np.empty(m), np.empty(m), np.zeros(m, dtype=np.uint8)
        device.launch("pow_eval", m, [x, np.array([kind, n], dtype=np.int32)], [exact, spec, flag])
        _, f = check_instance(kind, n, x, exact, spec, flag, cr, dist, hard=hard)
        off, total = off + f, total + m
    print(f"{KINDS[kind]} on the device: {total} arguments, {off} within {hard:.1e} ulp of a rounding "
          f"boundary and 1 ulp off")
    assert off <= total * 1e-3


GL_SRC = r"""
extern "C" __global__ void t_gl_pow_m(const double* x, const double* y, double* p, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  p[i] = inflx_gl_pow_m(x[i], y[0]);
}
"""
GL_HOST = r"""
#include <math.h>
void host_pow(const double* x, double y, double* p, long n) {
  for (long i = 0; i < n; i++) p[i] = pow(x[i], y);
}
"""


def test_glibc_flavour_per_point_pow_has_the_host_libm_bits(tmp_path):
    """inflx_gl_pow_m (flavour "glibc-all", class M) at every operand and literal exponent above:
    the host libm's bits, NaN for NaN."""
    import ctypes
    import subprocess

    from gpu_kernels import ROOT, Module
    from test_glibcmath import _has_fma, _host_glibc

    if not (_host_glibc() == "2.39" and _has_fma()):
        pytest.skip("bit identity is pinned to glibc 2.39's FMA ifunc variants")
    csrc = os.path.join(ROOT, "inflatox_b200", "csrc")
    src, so = tmp_path / "host_pow.c", tmp_path / "host_pow.so"
    src.write_text(GL_HOST)
    subprocess.run(["gcc", "-O2", "-fno-builtin", "-shared", "-fPIC", str(src), "-o", str(so), "-lm"],
                   check=True)  # fmt: skip
    lib = ctypes.CDLL(str(so))
    dp = ctypes.POINTER(ctypes.c_double)
    lib.host_pow.argtypes = [dp, ctypes.c_double, dp, ctypes.c_long]
    with open(os.path.join(csrc, "inflx_glibc_tables.cuh")) as fh:
        tables = fh.read()
    with open(os.path.join(csrc, "inflx_glibcmath.cuh")) as fh:
        header = fh.read().replace('#include "inflx_glibc_tables.cuh"', tables)
    mod = Module(header + GL_SRC)
    for kind in sorted(KINDS):
        for n in N_RANGE[kind]:
            x = arguments(kind, n)
            y = exponent(kind, n)
            d, h = np.empty(x.size), np.empty(x.size)
            mod.launch("t_gl_pow_m", x.size, [x, np.array([y], dtype=np.float64)], [d])
            lib.host_pow(x.ctypes.data_as(dp), y, h.ctypes.data_as(dp), x.size)
            bad = np.flatnonzero(~same_bits(d, h))
            assert bad.size == 0, (y, bad.size, x[bad[:3]], d[bad[:3]], h[bad[:3]])
