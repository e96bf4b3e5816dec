"""Randomly generated model artefacts: C text of random expression trees over x[0], x[1], args[k]
built ONLY from + - * / sqrt fabs and pow(.,2) - the operations this back-end claims to evaluate
bit-identically to the reference's CPU path.  The same text is compiled by gcc (reference flags,
driven by the oracle) and by the CUDA pipeline (Compiler.build_artifact: parser -> DAG -> rate
partition -> speculative division + slow path -> kernels).  Every finite value must agree to the
last bit, NaN/inf patterns must be identical - for the raw model functions and for the
arithmetic-only outputs of complete_analysis (consistency, eps_V, eps_H, omega)."""

import numpy as np
import pytest

import oracle
from inflatox_b200 import libinflx_rs as rs
from inflatox_b200.compiler import Compiler

pytestmark = pytest.mark.gpu

from raw_units import N_PAR, SPECIAL_UNIT, RawOracle as _RawOracle, make_unit  # noqa: E402


def _bit_identical(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    nan = np.isnan(a) & np.isnan(b)
    return (a.view(np.uint64) == b.view(np.uint64)) | nan | ((a == 0) & (b == 0))


@pytest.mark.parametrize("seed,conditionals", [(k, False) for k in range(12)] + [(k, True) for k in range(100, 110)])
def test_random_arithmetic_models_are_bit_identical(seed, conditionals, tmp_path):
    c_text = make_unit(seed, conditionals)
    orc = _RawOracle(c_text, str(tmp_path))
    comp = Compiler.__new__(Compiler)
    comp.nvrtc_opts = list(Compiler.default_nvrtc_flags)
    comp.output_path = str(tmp_path / "model.c")
    art_path = str(tmp_path / "model.bin")
    comp.build_artifact(c_text, art_path)
    lib = rs.open_inflx_dylib(art_path, False)
    lib.set_devices([0])
    rng = np.random.default_rng(seed)
    p = rng.uniform(0.5, 3.0, N_PAR)
    ext = (-2.0, 3.0, -1.5, 2.5)
    n0, n1 = 67, 139
    ss = np.array(ext).reshape(2, 2)
    # raw model functions
    v = np.zeros((n0, n1))
    lib.potential_array(v, p, ss)
    assert _bit_identical(v, orc.potential_array(p, n0, n1, ext)).all()
    h = lib.hesse_array(np.array([n0, n1]), p, ss)
    assert _bit_identical(h, orc.hesse_array(p, n0, n1, ext)).all()
    # closed forms: every output except delta (atan) and eta (tan) is pure IEEE arithmetic
    out = np.zeros((n0, n1, 6))
    rs.complete_analysis(lib, p, out, ss, False, 0)
    ref = orc.complete_analysis(p, n0, n1, ext)
    for k in (0, 1, 2, 5):
        same = _bit_identical(out[..., k], ref[..., k])
        assert same.all(), (seed, k, int((~same).sum()), out[..., k][~same][:3], ref[..., k][~same][:3])
    # delta = atan(.) and eta = omega*tan(delta) - 3 go through the atan/tan helper (<= 1 / 3 ulp)
    for k in (3, 4):
        assert (np.isnan(out[..., k]) == np.isnan(ref[..., k])).all()
        assert (np.isinf(out[..., k]) == np.isinf(ref[..., k])).all()
    fin = np.isfinite(ref[..., 4]) & np.isfinite(out[..., 4])
    assert (np.abs(out[..., 4][fin] - ref[..., 4][fin]) <= 4.5e-16 * np.abs(ref[..., 4][fin])).all()
    fin = np.isfinite(ref[..., 3]) & np.isfinite(out[..., 3])
    d_eta = np.abs(out[..., 3][fin] - ref[..., 3][fin])
    # tan amplifies the (<= 1 ulp) difference between two correctly working atan's by tan(delta)
    amp = 1.0 + np.abs(np.tan(ref[..., 4][fin]))
    assert (d_eta <= 1.5e-15 * amp * (np.abs(ref[..., 3][fin]) + 3.0)).all(), d_eta.max()
    c1 = np.zeros((n0, n1))
    rs.consistency_only(lib, p, c1, ss, False, 0)
    assert _bit_identical(c1, orc.consistency_only(p, n0, n1, ext)).all()
    ev = np.zeros((n0, n1))
    rs.epsilon_v_only(lib, p, ev, ss, False, 0)
    assert _bit_identical(ev, orc.epsilon_v_only(p, n0, n1, ext)).all()




@pytest.mark.parametrize(
    "params",
    [[1.0, 2.0, 3.0], [1e308, 0.0, 1e-320], [np.inf, -0.0, np.nan], [3e-310, 1e300, 5e-324]],
)
def test_irregular_operands_take_the_exact_path(params, tmp_path):
    """Zero, infinite, subnormal, huge and NaN denominators / numerators in every class (parameter,
    row, column, per point): the speculative division must hand these points to the IEEE slow
    path - results, including the signs of infinities, equal gcc's bit for bit."""
    orc = _RawOracle(SPECIAL_UNIT, str(tmp_path))
    comp = Compiler.__new__(Compiler)
    comp.nvrtc_opts = list(Compiler.default_nvrtc_flags)
    comp.output_path = str(tmp_path / "model.c")
    art_path = str(tmp_path / "model.bin")
    comp.build_artifact(SPECIAL_UNIT, art_path)
    lib = rs.open_inflx_dylib(art_path, False)
    lib.set_devices([0])
    p = np.array(params, dtype=np.float64)
    ext = (-1.0, 3.0, -2.0, 2.0)  # the grid contains x0 = 0, x0 = +-1, x1 = 0 and x0 = x1 exactly
    n0, n1 = 16, 32
    ss = np.array(ext).reshape(2, 2)

    def same(a, b):
        a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
        return (a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b)) | ((a == 0) & (b == 0))

    v = np.zeros((n0, n1))
    lib.potential_array(v, p, ss)
    ref = orc.potential_array(p, n0, n1, ext)
    assert same(v, ref).all(), (v[~same(v, ref)][:4], ref[~same(v, ref)][:4])
    h = lib.hesse_array(np.array([n0, n1]), p, ss)
    assert same(h, orc.hesse_array(p, n0, n1, ext)).all()
    out = np.zeros((n0, n1, 6))
    rs.complete_analysis(lib, p, out, ss, False, 0)
    ref = orc.complete_analysis(p, n0, n1, ext)
    for k in (0, 1, 2, 5):
        ok = same(out[..., k], ref[..., k])
        assert ok.all(), (k, out[..., k][~ok][:4], ref[..., k][~ok][:4])
    assert (np.isnan(out[..., 3:5]) == np.isnan(ref[..., 3:5])).all()
    assert (np.isinf(out[..., 3:5]) == np.isinf(ref[..., 3:5])).all()


@pytest.mark.parametrize(
    "params",
    [[1.0, 2.0, 3.0], [1e308, 0.0, 1e-320], [np.inf, -0.0, np.nan], [3e-310, 1e300, 5e-324]],
)
def test_constant_zero_v10_takes_the_special_epilogue_bit_for_bit(params, tmp_path):
    """GPU twin of the host-emulation test of the same name: a model whose v10 is the constant 0
    (the hyperinflation model's case) never divides by that zero, and still returns gcc's bits on
    every plane - consistency NaN everywhere, delta +0 / NaN, eta = omega * 0 - 3."""
    from raw_units import ZERO_V10_UNIT

    orc = _RawOracle(ZERO_V10_UNIT, str(tmp_path))
    comp = Compiler.__new__(Compiler)
    comp.nvrtc_opts = list(Compiler.default_nvrtc_flags)
    comp.output_path = str(tmp_path / "model.c")
    art_path = str(tmp_path / "model.bin")
    comp.build_artifact(ZERO_V10_UNIT, art_path)
    lib = rs.open_inflx_dylib(art_path, False)
    lib.set_devices([0])
    p = np.array(params, dtype=np.float64)
    ext, n0, n1 = (-1.0, 3.0, -2.0, 2.0), 16, 32
    out = np.zeros((n0, n1, 6))
    rs.complete_analysis(lib, p, out, np.array(ext).reshape(2, 2), False, 0)
    ref = orc.complete_analysis(p, n0, n1, ext)
    assert np.isnan(out[..., 0]).all() and np.isnan(ref[..., 0]).all()
    for k in (1, 2, 3, 4, 5):
        ok = _bit_identical(out[..., k], ref[..., k])
        assert ok.all(), (k, out[..., k][~ok][:4], ref[..., k][~ok][:4])
    assert (np.isinf(out) == np.isinf(ref)).all()


def _power_lib(c_text, tmp_path, libm="glibc"):
    comp = Compiler.__new__(Compiler)
    comp.nvrtc_opts = list(Compiler.default_nvrtc_flags)
    comp.libm = libm
    comp.output_path = str(tmp_path / "model.c")
    art_path = str(tmp_path / "model.bin")
    comp.build_artifact(c_text, art_path)
    lib = rs.open_inflx_dylib(art_path, False)
    lib.set_devices([0])
    return lib


def _within(name, got, ref, some_finite=True):
    import cases

    err, fin, nan_mm, inf_mm = cases.rel_err(got, ref)
    assert nan_mm == 0 and inf_mm == 0, (name, nan_mm, inf_mm)
    assert (fin.any() or not some_finite) and (err[fin] <= 1e-10).all(), (name, float(err[fin].max(initial=0)))


@pytest.mark.parametrize("scale", [1.0, 2.0**300, 2.0**-300, 2.0**345])
def test_per_point_literal_powers_across_overflow_and_underflow(scale, tmp_path):
    """GPU twin of the host-emulation test of the same name: per-point x^3, x^-3, x^7, x^1.5,
    x^-2.5, x^3.5, x^64 (double-double chains with the hardware seeds) of operands one grid carries
    past the overflow and subnormal thresholds - grid ops, the on-trajectory op and calc_V: NaN / inf
    masks of the oracle (glibc pow) and every finite value within 1e-10 of it."""
    from raw_units import POWER_EXTENT, POWER_UNIT

    orc = _RawOracle(POWER_UNIT, str(tmp_path))
    lib = _power_lib(POWER_UNIT, tmp_path)
    p = np.array([scale, 1.0, 1.0])
    ext, n0, n1 = POWER_EXTENT, 97, 131
    ss = np.array(ext).reshape(2, 2)
    v = np.zeros((n0, n1))
    lib.potential_array(v, p, ss)
    _within("potential_array", v, orc.potential_array(p, n0, n1, ext))
    _within("hesse_array", lib.hesse_array(np.array([n0, n1]), p, ss), orc.hesse_array(p, n0, n1, ext))
    out = np.zeros((n0, n1, 6))
    rs.complete_analysis(lib, p, out, ss, False, 0)
    _within("complete_analysis", out, orc.complete_analysis(p, n0, n1, ext))
    rng = np.random.default_rng(64)
    xs = np.ascontiguousarray(np.stack([rng.uniform(ext[0], ext[1], 777), rng.uniform(ext[2], ext[3], 777)], 1))
    traj = np.zeros((xs.shape[0], 6))
    rs.complete_analysis_on_trajectory(lib, p, xs, traj, False, 0)
    _within("complete_analysis_on_trajectory", traj, orc.complete_analysis_on_trajectory(p, xs))
    calc_v = np.array([lib.potential(x, p) for x in xs[:64]])
    _within("calc_V", calc_v, np.array([orc.potential(x, p) for x in xs[:64]]), some_finite=False)
    if scale == 2.0**345:
        assert np.isinf(v).any() and np.isfinite(v).any()


def test_row_class_literal_powers_in_the_correctly_rounded_flavour(tmp_path):
    """libm="cr": powers of x[0] alone through the same chains in the row pre-pass, across the
    thresholds: NaN / inf masks of the oracle and every finite point within 1e-10 of it."""
    from raw_units import POWER_EXTENT, POWER_ROW_UNIT

    orc = _RawOracle(POWER_ROW_UNIT, str(tmp_path))
    lib = _power_lib(POWER_ROW_UNIT, tmp_path, libm="cr")
    ext, n0, n1 = POWER_EXTENT, 101, 37
    for scale in (1.0, 2.0**300, 2.0**-300, 2.0**345):
        p = np.array([scale, 1.0, 1.0])
        out = np.zeros((n0, n1, 6))
        rs.complete_analysis(lib, p, out, np.array(ext).reshape(2, 2), False, 0)
        _within(f"complete_analysis scale {scale}", out, orc.complete_analysis(p, n0, n1, ext))
