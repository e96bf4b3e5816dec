"""`Compiler` / printers: the string-level pins of the reference's tests/test_compiler.py:25-82,
plus: generated C identical to the reference's own output, GSL rejection, artefact container."""
import os
import re

import pytest
import sympy

import cases
import oracle
import inflatox_b200 as ix
from inflatox_b200.compiler import (
    CInflatoxPrinter,
    GSLInflatoxPrinter,
    UnsupportedFunctionError,
    nvrtc_compile,
    read_artifact_metadata,
)


@pytest.fixture
def cprinter():
    x, y, a, b, xdot, ydot = sympy.symbols("x y a b \\dot{{x}} \\dot{{y}}")
    return CInflatoxPrinter([x, y], [xdot, ydot])


@pytest.fixture
def gslprinter():
    x, y, a, b, xdot, ydot = sympy.symbols("x y a b \\dot{{x}} \\dot{{y}}")
    return GSLInflatoxPrinter([x, y], [xdot, ydot])


def test_cinflatox_printer(cprinter):
    x, y, a, b, xdot, ydot = sympy.symbols("x y a b \\dot{{x}} \\dot{{y}}")
    assert "x[0]" == cprinter._print_Symbol(x)
    assert "x[1]" == cprinter._print_Symbol(y)
    assert "args[0]" == cprinter._print_Symbol(a)
    assert "args[1]" == cprinter._print_Symbol(b)
    assert "xdot[0]" == cprinter._print_Symbol(xdot)
    assert "xdot[1]" == cprinter._print_Symbol(ydot)
    assert "pow(x[0], 2) + x[1]" == cprinter.doprint(x**2 + y)
    assert "x[0]*x[1]" == cprinter.doprint(x * y)
    assert "sqrt(args[0])*x[1]" == cprinter.doprint(sympy.sqrt(a) * y)
    assert "sin(x[0])" == cprinter.doprint(sympy.sin(x))


def test_gslinflatox_printer_headers(gslprinter):
    x, y = sympy.symbols("x y")
    gslprinter.doprint(sympy.besselj(1, x))
    assert gslprinter.BESSELH in gslprinter.required_headers
    gslprinter.doprint(sympy.hyper([], [1], x))
    assert gslprinter.HYPERH in gslprinter.required_headers


def test_gslinflatox_bessel(gslprinter):
    x, y, n = sympy.symbols("x y n")
    assert "gsl_sf_bessel_J0(x[0])" == gslprinter.doprint(sympy.besselj(0, x))
    assert "gsl_sf_bessel_J1(x[0])" == gslprinter.doprint(sympy.besselj(1, x))
    assert "gsl_sf_bessel_Jn(10, x[0])" == gslprinter.doprint(sympy.besselj(10, x))
    assert "gsl_sf_bessel_Jnu(0.50000000000000000, x[0])" == gslprinter.doprint(
        sympy.besselj(0.5, x)
    )


def test_gslinflatox_hyper(gslprinter):
    x, y, n = sympy.symbols("x y n")
    assert "gsl_sf_hyperg_2F0(0, 1, x[0])" == gslprinter.doprint(sympy.hyper([0, 1], [], x))
    assert "gsl_sf_hyperg_2F1(0, 1, 2, x[0])" == gslprinter.doprint(sympy.hyper([0, 1], [2], x))
    assert "gsl_sf_hyperg_1F1(0, 1, x[0])" == gslprinter.doprint(sympy.hyper([0], [1], x))
    assert "gsl_sf_hyperg_0F1(0, x[0])" == gslprinter.doprint(sympy.hyper([], [0], x))
    with pytest.raises(Exception) as exinfo:
        gslprinter.doprint(sympy.hyper([0, 3, 4], [1, 2], x))
    assert "Cannot compute" in str(exinfo.value)


# ------------------------------------------------------------------------------------------------
def _functions(text: str) -> dict[str, str]:
    out = {}
    for m in re.finditer(r"^(?:double|void) (\w+)\([^)]*\)\{\n(.*?)\n\}", text, re.S | re.M):
        out[m.group(1)] = m.group(2)
    return out


HOT = ["V", "inner_prod", "v00", "v01", "v10", "v11", "v", "w1", "grad_norm_squared"]


@pytest.mark.parametrize("model", cases.MODELS)
def test_generated_c_equals_the_references_output(model):
    """Same functions, same text, same `args[k]` numbering as the unmodified reference compiler
    produced for the same symbolic model (fixture: tests/golden/c, made by make_golden.py).  The
    eom* functions are excluded: they are off the path, and sympy re-distributes their leading
    -1/2 when the model fixture is un-pickled."""
    m = cases.load_model(model)
    meta = oracle.golden_meta(model)
    comp = ix.Compiler(m, silent=True, cse=meta["cse"])
    mine, gold = _functions(comp._generate_c_source()), _functions(oracle.golden_c_text(model))
    os.remove(comp.output_path)
    for fn in HOT:
        assert mine[fn] == gold[fn], f"{model}: function {fn} differs from the reference's text"
    assert comp.symbol_dict == meta["symbol_dictionary"]
    assert set(mine) == set(gold)


def test_compile_produces_a_cuda_artefact():
    art = cases.artifact("angular")
    assert isinstance(art, ix.CompilationArtifact)
    assert art.n_fields == 2 and art.n_parameters == 3
    assert art.symbol_dictionary["phi"] == "x[0]" and art.symbol_dictionary["alpha"] == "args[0]"
    assert art.lookup_symbol(sympy.Symbol("m_chi")) == "args[1]"
    meta = read_artifact_metadata(art.shared_object_path)
    assert meta["abi_version"] == (5, 0, 0) and meta["model_name"] == "angular"
    assert not meta["fmad"] and meta["rows_per_thread"] >= 1
    assert "--gpu-architecture=sm_100a" in meta["nvrtc_options"]
    assert set(meta["groups"]) == {"cmp", "con", "eps", "bas", "pot", "hes"}
    assert meta["flops_per_point"]["complete_analysis"] == art.flops_per_point()
    with open(art.shared_object_path, "rb") as fh:
        blob = fh.read()
    assert blob[:8] == b"INFLXB2\0" and b"\x7fELF" in blob  # cubins are ELF images


def test_artifact_is_removed_with_auto_cleanup():
    m = cases.load_model("doc")
    art = ix.Compiler(m, silent=True, cleanup=True).compile()
    path = art.shared_object_path
    assert os.path.exists(path)
    del art
    assert not os.path.exists(path)


def test_gsl_special_functions_are_rejected_at_compile_time():
    m = cases.load_model("doc")
    r = m.coordinates[0]
    m.potential = m.potential + sympy.besselj(0, r)
    with pytest.raises(UnsupportedFunctionError, match="no fp64 device implementation"):
        ix.Compiler(m, silent=True, link_gsl=True).compile()


def test_nvrtc_errors_surface_the_log():
    with pytest.raises(Exception, match="NVRTC compilation"):
        nvrtc_compile("__global__ void k() { this is not C++ }", "bad.cu",
                      ["--gpu-architecture=sm_100a"], use_cache=False)  # fmt: skip


def test_flops_per_point_are_frozen():
    """F(model, op) of SURVEY.md 8(d), recomputed from the emitted DAG; frozen here so a code
    generator change that alters the roofline numerator is noticed."""
    want = {"doc": 102, "hyper": 59, "angular": 244, "egno": 587, "d5": 889}
    for model, f in want.items():
        assert cases.artifact(model).flops_per_point("complete_analysis") == f
    assert cases.artifact("angular").flops_per_point("consistency_only") == 205


def test_piecewise_models_compile():
    """sympy prints Piecewise / sign / Heaviside as (multi-line) C conditionals; the parser, the
    DAG and the CUDA emitter carry them (cmp / and / or / not / sel nodes)."""
    m = cases.load_model("doc")
    r, th = m.coordinates
    m.potential = m.potential + sympy.Piecewise((r**2, r > 1), (sympy.sign(th) * th, True))
    comp = ix.Compiler(m, silent=True)
    art = comp.compile()
    assert "?" in comp.c_source and art.n_parameters == 1
    assert read_artifact_metadata(art.shared_object_path)["flops_per_point"]["potential"] > 7


def test_a_cubin_cache_that_cannot_be_written_is_still_used(tmp_path, monkeypatch):
    """A cache shipped pre-filled in a read-only tree: a cubin it holds is loaded, one it lacks is
    compiled and returned (and reused within the process) instead of failing on the write."""
    from inflatox_b200 import compiler

    monkeypatch.setenv("INFLATOX_CACHE_DIR", str(tmp_path))
    opts = ["--gpu-architecture=sm_100a", "--std=c++17"]
    src = f'extern "C" __global__ void k(double* p) {{ p[0] = 2.0; }}  // {tmp_path.name}'
    shipped = nvrtc_compile(src, "k.cu", opts)  # writable: stored
    assert len(list(tmp_path.glob("*.cubin"))) == 1

    def read_only(*args, **kwargs):
        raise PermissionError(13, "Permission denied")

    monkeypatch.setattr(compiler.os, "replace", read_only)
    assert nvrtc_compile(src, "k.cu", opts) == shipped
    other = src.replace("2.0", "3.0")
    a = nvrtc_compile(other, "k.cu", opts)
    assert a and a != shipped
    assert sorted(p.name for p in tmp_path.iterdir()) == [p.name for p in tmp_path.glob("*.cubin")]
    assert len(list(tmp_path.glob("*.cubin"))) == 1  # nothing stored, no temporary left behind
    assert nvrtc_compile(other, "k.cu", opts) == a
