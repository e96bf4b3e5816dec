"""Raw C model units for tests: a random generator over the operations the CUDA back-end claims to
evaluate bit-identically (+ - * / sqrt fabs pow(.,2), comparisons, && || !, ?:), and an oracle
front-end that compiles any such unit with gcc and the reference's flag set."""
import ctypes
import os
import random
import subprocess

import oracle

N_PAR = 3
PREAMBLE = """#include <math.h>
#include <stdint.h>
const uint16_t VERSION[3] = {5,0,0};
const uint32_t DIM = 2;
const uint32_t N_PARAMETERS = %d;
char *const MODEL_NAME = "random%d";
const char USE_GSL = 0;

"""


def rand_cond(rng: random.Random, depth: int) -> str:
    a, b = rand_expr(rng, depth - 1, False), rand_expr(rng, depth - 1, False)
    c = f"{a} {rng.choice(['<', '>', '<=', '>=', '==', '!='])} {b}"
    r = rng.random()
    if r < 0.2:
        return f"{c} && {rand_expr(rng, 1, False)} > 0"
    if r < 0.35:
        return f"{c} || !({rand_expr(rng, 1, False)} < 1)"
    return c


def rand_expr(rng: random.Random, depth: int, conditionals: bool = False) -> str:
    if depth <= 0 or rng.random() < 0.15:
        r = rng.random()
        if r < 0.35:
            return "x[0]"
        if r < 0.7:
            return "x[1]"
        if r < 0.85:
            return f"args[{rng.randrange(N_PAR)}]"
        return rng.choice(["2", "3", "0.5", "1.25", "7", "(1.0/3.0)", "10"])
    r = rng.random()
    if conditionals and r < 0.18:
        a, b = rand_expr(rng, depth - 1, True), rand_expr(rng, depth - 1, True)
        if rng.random() < 0.3:  # sympy's sign(): difference of two comparisons
            return f"({a})*((({b}) > 0) - (({b}) < 0))"
        return f"(({rand_cond(rng, 2)}) ? (\n   {a}\n)\n: (\n   {b}\n))"
    a, b = rand_expr(rng, depth - 1, conditionals), rand_expr(rng, depth - 1, conditionals)
    if r < 0.25:
        return f"({a} + {b})"
    if r < 0.45:
        if a == b:
            # x - x is an exact zero whose SIGN the reference's -fno-signed-zeros leaves to the
            # compiler (and 1/+-0 then differs in the sign of infinity): not a parity question
            b = f"({b} + 1)"
        return f"({a} - {b})"
    if r < 0.7:
        return f"({a})*({b})"
    if r < 0.88:
        return f"({a})/({b})"
    if r < 0.94:
        return f"sqrt(fabs({a}) + 0.125)"
    if r < 0.97:
        return f"sqrt({a})"  # may be NaN: legit
    return f"pow({a}, 2)"


def make_unit(seed: int, conditionals: bool = False) -> str:
    rng = random.Random(seed)
    xa = "(const double x[], const double args[])"
    text = PREAMBLE % (N_PAR, seed)
    for name in ("V", "v00", "v01", "v10", "v11", "grad_norm_squared"):
        body = rand_expr(rng, rng.randint(3, 6), conditionals)
        text += f"double {name}{xa}{{\n    return {body};\n}}\n\n"
    text += (
        "double inner_prod(const double x[], const double args[], const double v1[], "
        "const double v2[]){\n    const double g00 = 1;\n    const double g11 = 1;\n"
        "    return 0.0 + (g00 * v1[0] * v2[0]) + (g11 * v1[1] * v2[1]);\n}\n\n"
    )
    for name in ("v", "w1"):
        text += (
            f"void {name}(const double x[], const double args[], double v_out[]){{\n"
            f"    v_out[0] = {rand_expr(rng, 3, conditionals)};\n"
            f"    v_out[1] = {rand_expr(rng, 3, conditionals)};\n    return;\n}}\n\n"
        )
    return text


# zero / inf / subnormal / huge / NaN operands in every class (parameter, row, column, point)
SPECIAL_UNIT = PREAMBLE % (N_PAR, 999) + """
double V(const double x[], const double args[]){
    return (x[1] + 2)/(x[0]) + (x[1])/(args[0]*x[0]) + (x[0])/(x[1]);
}
double v00(const double x[], const double args[]){
    return (x[1])/(args[1]) + sqrt(x[0] - 1)*x[1];
}
double v01(const double x[], const double args[]){
    return (x[1]*x[0])/(args[2]);
}
double v10(const double x[], const double args[]){
    return (x[0] - x[1])/((x[0])*(x[0]) - 1);
}
double v11(const double x[], const double args[]){
    return (1.0/3.0)/(x[1]) + (x[0])/(args[0]);
}
double grad_norm_squared(const double x[], const double args[]){
    return ((x[1])/(x[0]))/(x[1] - x[0]);
}
double inner_prod(const double x[], const double args[], const double v1[], const double v2[]){
    const double g00 = 1;
    const double g11 = 1;
    return 0.0 + (g00 * v1[0] * v2[0]) + (g11 * v1[1] * v2[1]);
}
void v(const double x[], const double args[], double v_out[]){
    v_out[0] = x[0];
    v_out[1] = x[1];
    return;
}
void w1(const double x[], const double args[], double v_out[]){
    v_out[0] = x[1];
    v_out[1] = x[0];
    return;
}
"""


class RawOracle(oracle.Oracle):
    """oracle driver over an arbitrary generated C unit (same reference flag set)."""

    def __init__(self, c_text: str, workdir: str):
        src = os.path.join(workdir, "model.c")
        so = os.path.join(workdir, "model.so")
        with open(src, "w") as fh:
            fh.write(c_text)
        flags = [f for f in oracle.REFERENCE_FLAGS if f != "-Werror"]
        subprocess.run(["gcc", "-o", so, src, *flags, "-ffp-contract=off"], check=True)
        b = oracle._Build()
        self.quad, self.sfx = False, ""
        self.lib = ctypes.CDLL(b.driver(False))
        self.path, self.h = so, ctypes.c_void_p()
        fn = self.lib.oracle_open
        fn.restype = ctypes.c_int
        assert fn(so.encode(), ctypes.byref(self.h)) == 0
        self.n_fields, self.n_params, self.meta = 2, N_PAR, {}


# the same unit with v10 == 0: a Hesse matrix diagonal in the {v, w} basis (the README's
# hyperinflation model has it).  complete_analysis then takes the closed special form
# inflx_op_complete_v10z_s; irregular operands must come out as gcc's x / 0, 0 / x, inf * 0 do.
ZERO_V10_UNIT = SPECIAL_UNIT.replace(
    "    return (x[0] - x[1])/((x[0])*(x[0]) - 1);", "    return 0;"
).replace('random999', 'zero_v10')
assert "return 0;" in ZERO_V10_UNIT


# per-point literal powers (exponents 3, -3, 7, 1.5, -2.5, 3.5, 64) of expressions in x[0], x[1] and
# args[0]: the generator emits the double-double chains inflx_powi / inflx_powi_neg / inflx_powh /
# inflx_powh_neg.  With args[0] = 2^300, 2^-300 or 2^345 and x[0] x[1] spanning 2^-20 .. 2^4 on the
# grid, one grid crosses the overflow, subnormal and zero thresholds of the powers.
POWER_UNIT = PREAMBLE % (N_PAR, 64) + """
double V(const double x[], const double args[]){
    return pow(args[0]*x[0]*x[1], 3) + pow(x[0]*x[1], 64);
}
double v00(const double x[], const double args[]){
    return pow(args[0]*(x[0] + x[1]*x[1]), -3);
}
double v01(const double x[], const double args[]){
    return x[0]*x[1];
}
double v10(const double x[], const double args[]){
    return pow(x[0]*x[1]*args[0], 7) - pow(args[0]*x[0] + x[1], 1.5);
}
double v11(const double x[], const double args[]){
    return pow(args[0]*x[0]*x[1] + x[1], -2.5);
}
double grad_norm_squared(const double x[], const double args[]){
    return pow(args[0]*x[1] + x[0], 3.5);
}
double inner_prod(const double x[], const double args[], const double v1[], const double v2[]){
    const double g00 = 1;
    const double g11 = 1;
    return 0.0 + (g00 * v1[0] * v2[0]) + (g11 * v1[1] * v2[1]);
}
void v(const double x[], const double args[], double v_out[]){
    v_out[0] = x[0];
    v_out[1] = x[1];
    return;
}
void w1(const double x[], const double args[], double v_out[]){
    v_out[0] = x[1];
    v_out[1] = x[0];
    return;
}
"""
POWER_SCALES = (1.0, 2.0**300, 2.0**-300, 2.0**345)
POWER_EXTENT = (0.001, 4.0, 0.001, 4.0)

# flavour "cr": powers of x[0] alone are evaluated once per grid row, by the same chains
POWER_ROW_UNIT = POWER_UNIT.replace("random64", "powrow").replace(
    "return pow(args[0]*x[0]*x[1], 3) + pow(x[0]*x[1], 64);",
    "return pow(args[0]*x[0], 3) + pow(x[0], 64) + x[1];").replace(
    "return pow(args[0]*(x[0] + x[1]*x[1]), -3);", "return pow(args[0]*x[0], -3) + x[1];").replace(
    "return pow(args[0]*x[0]*x[1] + x[1], -2.5);", "return pow(args[0]*x[0], -2.5) + x[1];")
assert POWER_ROW_UNIT.count(" + x[1];") == 3
