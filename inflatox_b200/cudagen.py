"""CUDA code generator: one hash-consed model DAG (`cexpr.Dag`) -> sm_100a kernels.

The reference evaluates five separately compiled C functions per grid point (reference
src/anguelova.rs:110-119 -> src/hesse_bindings.rs:54-58, 213-231), each recomputing the metric,
the Christoffel symbols and the gradient norm from scratch.  Here every function of the model
lives in ONE DAG and each DAG node is evaluated once, at the *lowest rate at which it changes*:

    class P  depends on the model parameters only        -> once per parameter vector
    class R  depends on x[0] (and parameters)            -> once per grid ROW      (`inflx_rows`)
    class C  depends on x[1] (and parameters)            -> once per thread (= per grid column,
                                                            reused over INFLX_RPT rows)
    class M  depends on both coordinates                 -> once per grid point

A value crosses from a slower class to a faster one through a *frontier*: P-frontier values sit
in `__constant__` memory (so they are free operands of the FP64 instructions), R-frontier values in
a small global array `rc[row][k]` that every thread of a row reads with warp-uniform loads.  The
operations, their operands and their order are exactly those of the C text, so hoisting changes
no rounding: a node is the same IEEE operation wherever it is evaluated.

For the test models this moves most of the work off the per-point path (d5: 911 DAG nodes, 169 of
them class M; EGNO: 618 / 193), including every log / general pow.

Kernels are generated per *group* of output functions (one cubin each), so an operation never
pays for model functions it does not read:

    cmp  V v00 v10 v11 |grad V|^2   complete_analysis (+ on-trajectory)
    con  V v00 v10 v11              consistency_only, consistency_rapidturn_only (+ on-trajectory)
    eps  V |grad V|^2               epsilon_v_only (+ on-trajectory)
    bas  v (and w1, inner_prod)     flag_quantum_dif; basis validation
    pot  V                          potential / potential_array
    hes  v00 v01 v10 v11            hesse / hesse_array
"""
from __future__ import annotations

import math
import os

from .cexpr import Dag, ParsedUnit

_CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")

# resident CTAs per SM the register allocation of a group's grid kernels must allow (128-thread
# CTAs: 4 -> 128 registers, 5 -> 96, 6 -> 80).  From the tools/tune.py sweeps over the five test
# models: the six-output kernels are fastest at 6, the single-plane ones at 5 - unless the model
# keeps many column-class values live across the row loop (2 registers each for the whole loop):
# then the cap spills them to local memory, 6 CTAs x 128 threads x 200 B no longer fit L1 and the
# reloads stall (angular: 27 values, 224 B of stack at 80 registers; tools/ab.py round 2:
# complete_analysis 16384^2 6.18 -> 5.88 ms at 4 CTAs/SM, consistency_only 4096^2 0.249 -> 0.242).
# `GroupProgram.min_blocks` lowers the count until 2 * (live column values) + WORKING_REGS fits.
MIN_BLOCKS = {"cmp": 6, "hes": 6}
REGS_AT = {6: 80, 5: 96, 4: 128}
WORKING_REGS = 48
PC_CAPACITY = 7680  # doubles of __constant__ memory for P-frontier values (60 of the 64 KiB)
MAX_FAST_POW = 64  # |exponent| up to which literal (half-)integer powers use the dd chains
# libm flavours for the model's libm calls in the hoisted node classes P / R / C (a column block
# that contains such a call is evaluated by the `inflx_cols` pre-pass, once per column, instead of
# once per CTA in the grid kernel's prologue):
#   "glibc"  (default) csrc/inflx_glibcmath.cuh: the algorithm glibc 2.39 runs on the reference's
#            host, bit for bit - the reference's own result (compiler.py:299-310 links -lm).  Also
#            used for pow(x, n) with a literal n in those classes, because glibc's pow is not always
#            correctly rounded and the dd chains are.  60-100 FP64 instructions per call.
#   "cr"     csrc/inflx_crmath.cuh: correctly rounded in double-double arithmetic (~1000 FP64
#            instructions per call); literal powers through the correctly rounded dd chains.
#   "device" libdevice everywhere (1-2 ulp).
# Per grid point (class M) a libm call uses libdevice and a literal (half-)integer power the
# correctly rounded dd chain (EGNO: pow(., -0.5), pow(., 1.5); d5: pow(., 1.5)) - except in flavour
#   "glibc-all" = "glibc" + the class-M calls of GL_FUNCTIONS through inflx_gl_* as well (bit
#            identity with the reference wherever glibc's pow misrounds, at 60-100 FP64
#            instructions and an out-of-line call per point; measured in DESIGN.md).
LIBM_FLAVOURS = ("glibc", "glibc-all", "cr", "device")
GL_FUNCTIONS = ("pow", "log", "exp", "expm1", "sin", "cos", "tanh")
CR_FUNCTIONS = ("pow", "log", "exp", "sin", "cos")
CR_CLASSES = ("P", "R", "C")

# fixed epilogue cost in flops (SURVEY.md 8a: a8 as written = 46, a9 = 13; the rest counted the
# same way: + - * / sqrt and every libm-class call = 1, abs/neg/compare = 0)
EPILOGUE_FLOPS = {
    "complete_analysis": 46,
    "consistency_only": 13,
    "consistency_rapidturn_only": 8,
    "epsilon_v_only": 3,
    "flag_quantum_dif": 0,
    "potential": 0,
    "hesse": 0,
    "basis": 0,
}

# group -> (grid roots, extra point-only roots, grid ops, point ops)
GROUPS = {
    "cmp": (("V", "v00", "v10", "v11", "g2"), (), ("complete_analysis",), ("complete_analysis",)),
    "con": (
        ("V", "v00", "v10", "v11"),
        (),
        ("consistency_only", "consistency_rapidturn_only"),
        ("consistency_only", "consistency_rapidturn_only"),
    ),
    "eps": (("V", "g2"), (), ("epsilon_v_only",), ("epsilon_v_only",)),
    "bas": (("b0", "b1"), ("w0", "w1", "ip"), ("flag_quantum_dif",), ("basis",)),
    "pot": (("V",), (), ("potential",), ("potential",)),
    "hes": (("v00", "v01", "v10", "v11"), (), ("hesse",), ("hesse",)),
}

# point ops that additionally get a one-launch scalar kernel (`inflx_scalar_<op>`)
SCALAR_OPS = ("potential", "hesse")


def _lit(v: float) -> str:
    if math.isnan(v):
        return "(0.0/0.0)"
    if math.isinf(v):
        return "(1.0/0.0)" if v > 0 else "(-1.0/0.0)"
    s = repr(float(v))
    if "e" not in s and "." not in s and "n" not in s:
        s += ".0"
    return f"({s})" if v < 0 or (v == 0 and math.copysign(1, v) < 0) else s


def _int_pow_mults(n: int) -> int:
    n = abs(n)
    if n <= 1:
        return 0
    return n.bit_length() - 1 + bin(n).count("1") - 1


class ModelRoots:
    """Names the DAG nodes of the model functions the hot path reads (reference
    src/hesse_bindings.rs:195-232 `fns[0]=v00, fns[2]=v10, fns[3]=v11`; dylib.rs:163-183)."""

    def __init__(self, unit: ParsedUnit):
        f = unit.functions
        need = ["V", "v00", "v01", "v10", "v11", "grad_norm_squared", "v", "w1", "inner_prod"]
        missing = [n for n in need if n not in f]
        if missing:
            raise Exception(f"model source lacks the function(s) {missing}; is it a 2-field model?")
        self.node = {
            "V": f["V"].result,
            "v00": f["v00"].result,
            "v01": f["v01"].result,
            "v10": f["v10"].result,
            "v11": f["v11"].result,
            "g2": f["grad_norm_squared"].result,
            "b0": f["v"].outputs[0],
            "b1": f["v"].outputs[1],
            "w0": f["w1"].outputs[0],
            "w1": f["w1"].outputs[1],
            "ip": f["inner_prod"].result,
        }


class GroupProgram:
    """Classification, frontiers, flop counts and CUDA text for one group of model functions.

    Works on a *local* node table: the DAG nodes reachable from the group's roots plus one
    pseudo-node ("rcp", b) per distinct denominator b of a division.  ("rcp", b) stands for the
    refined reciprocal `inflx_rcp_s(b)` the speculative division needs; being a node, it is
    classified and hoisted like any other value, so a per-point quotient by a row- or
    parameter-class denominator costs 3 FP64 instructions instead of 9.
    """

    def __init__(self, dag: Dag, roots: ModelRoots, group: str, n_params: int, libm: str = "glibc",
                 cols: str = "auto", store: str = "auto"):
        if libm not in LIBM_FLAVOURS:
            raise Exception(f"unknown libm flavour {libm!r}: one of {LIBM_FLAVOURS}")
        if cols not in ("auto", "always", "never"):
            raise Exception(f"unknown column pre-pass mode {cols!r}: auto, always or never")
        self.cols = cols
        if store not in ("auto", "transposed", "direct"):
            raise Exception(f"unknown store mode {store!r}: auto, transposed or direct")
        self.store = store
        self.dag = dag
        self.group = group
        self.n_params = n_params
        self.libm = libm
        grid_names, point_names, self.grid_ops, self.point_ops = GROUPS[group]
        self.grid_roots = {n: roots.node[n] for n in grid_names}
        self.point_roots = {n: roots.node[n] for n in grid_names + point_names}
        self.extra: dict[int, tuple] = {}  # pseudo-nodes, ids >= len(dag.nodes)
        self.rcp_of: dict[int, int] = {}  # denominator node -> its ("rcp", b) pseudo-node
        self.all_nodes = self._with_reciprocals(dag.reachable(self.point_roots.values()))
        grid_plain = set(dag.reachable(self.grid_roots.values()))
        self.grid_nodes = [
            i
            for i in self.all_nodes
            if i in grid_plain or (i in self.extra and self._rcp_used_by_grid(i, grid_plain))
        ]
        self._classify()
        self._frontiers()

    # -- local node table ----------------------------------------------------------------------
    def node(self, i: int) -> tuple:
        return self.extra[i] if i in self.extra else self.dag.nodes[i]

    def operands(self, i: int) -> tuple[int, ...]:
        n = self.node(i)
        if n[0] == "rcp":
            return (n[1],)
        ops = self.dag.operands(i)
        if n[0] == "/" and n[2] in self.rcp_of:
            return ops + (self.rcp_of[n[2]],)
        return ops

    def _with_reciprocals(self, nodes: list[int]) -> list[int]:
        out = []
        next_id = len(self.dag.nodes)
        for i in nodes:
            n = self.dag.nodes[i]
            if n[0] == "/" and n[2] not in self.rcp_of:
                self.extra[next_id] = ("rcp", n[2])
                self.rcp_of[n[2]] = next_id
                out.append(next_id)  # topological: right before its first user
                next_id += 1
            out.append(i)
        return out

    def _rcp_used_by_grid(self, r: int, grid_plain: set) -> bool:
        b = self.extra[r][1]
        return any(
            self.dag.nodes[i][0] == "/" and self.dag.nodes[i][2] == b for i in grid_plain
        )

    # -- analysis ----------------------------------------------------------------------------
    def _classify(self):
        dep: dict[int, int] = {}
        for i in self.all_nodes:
            n = self.node(i)
            k = n[0]
            if k == "x":
                if n[1] > 1:
                    raise Exception("the CUDA back-end evaluates 2-field models only")
                dep[i] = 2 << n[1]
            elif k == "p":
                dep[i] = 1
            elif k in ("v1", "v2"):
                dep[i] = 8
            elif k in ("c", "i"):
                dep[i] = 0
            elif k == "xd":
                raise Exception("field velocities are not part of the grid-evaluation path")
            else:
                b = 0
                for o in self.operands(i):
                    b |= dep[o]
                dep[i] = b
        self.dep = dep

    def klass(self, i: int) -> str:
        m = self.dep[i]
        if m & 8:
            return "V"
        if m == 0:
            # an unfoldable call on constants (e.g. tgamma(2.5)) is evaluated with the parameters
            return "P" if self.is_op(i) else "K"
        if m == 1:
            return "P"
        if m in (2, 3):
            return "R"
        if m in (4, 5):
            return "C"
        return "M"

    def _frontiers(self):
        users: dict[int, list[int]] = {}
        for i in self.all_nodes:
            for o in self.operands(i):
                users.setdefault(o, []).append(i)
        self.users = users
        root_ids = set(self.point_roots.values())
        self.p_frontier = [
            i
            for i in self.all_nodes
            if self.klass(i) == "P"
            and (i in root_ids or any(self.klass(u) != "P" for u in users.get(i, ())))
        ]
        grid_set = set(self.grid_nodes)
        grid_root_ids = set(self.grid_roots.values())
        self.r_frontier = [
            i
            for i in self.grid_nodes
            if self.klass(i) == "R"
            and (
                i in grid_root_ids
                or any(u in grid_set and self.klass(u) != "R" for u in users.get(i, ()))
            )
        ]
        if len(self.p_frontier) > PC_CAPACITY:
            raise Exception(
                f"model needs {len(self.p_frontier)} parameter-class values per vector; the "
                f"__constant__ bank holds {PC_CAPACITY}"
            )
        self.p_slot = {n: k for k, n in enumerate(self.p_frontier)}
        self.r_slot = {n: k for k, n in enumerate(self.r_frontier)}
        # column pre-pass: only when the column block is expensive (holds a correctly rounded
        # libm call); a cheap column block stays in the grid kernel's prologue
        self.cols_prepass = any(
            self.klass(i) == "C" and self.node(i)[0] == "f" and self._hoisted_libm(i) is not None
            for i in self.grid_nodes
        )
        if self.cols != "auto":
            self.cols_prepass = self.cols == "always" and any(
                self.klass(i) == "C" and self.is_op(i) for i in self.grid_nodes
            )
        # column-class values the per-point code reads: live in registers over the whole row loop
        self.c_live = [
            i
            for i in self.grid_nodes
            if self.klass(i) == "C"
            and self.is_op(i)
            and (
                i in grid_root_ids
                or any(u in grid_set and self.klass(u) != "C" for u in users.get(i, ()))
            )
        ]
        self.c_frontier = self.c_live if self.cols_prepass else []
        # complete_analysis kernels with very little arithmetic per 48-byte record are bound by the
        # L1 -> L2 store path, not by issue slots: they use the warp-transposed store
        # (inflx_store6_warp).  Estimate: ~2.5 issue cycles per FP64 instruction (tools/sass_cost.py)
        # against the ~270 cycles per warp and row the HBM write roof allows.
        self.transposed_store = self.group == "cmp" and (
            self.store == "transposed"
            or (self.store == "auto" and self._estimated_fp64_per_point() * 2.5 < 270)
        )
        self.min_blocks = MIN_BLOCKS.get(self.group, 5)
        while self.min_blocks > 4 and 2 * len(self.c_live) + WORKING_REGS > REGS_AT[self.min_blocks]:
            self.min_blocks -= 1
        self.c_slot = {n: k for k, n in enumerate(self.c_frontier)}
        # rows of the row-frontier array are read with 128-bit loads: keep them 16-byte aligned
        self.n_row_slots = (len(self.r_frontier) + 1) & ~1

    def _estimated_fp64_per_point(self) -> int:
        """Rough FP64 instruction count of one grid point of complete_analysis: class-M operations
        (a quotient 3, its own reciprocal 5, a square root 9) + the epilogue (160; 60 in the closed
        form for a constant-zero v10)."""
        n = 0
        for i in self.nodes_of("M", self.grid_nodes):
            k = self.node(i)[0]
            n += {"/": 3, "rcp": 5}.get(k, 1)
            if k == "f":
                n += 8 if self.node(i)[1] == "sqrt" else 20
        return n + (60 if self._v10_is_plus_zero() else 160)

    def _hoisted_libm(self, i: int) -> str | None:
        """Prefix of the out-of-line libm function ("inflx_gl_" / "inflx_cr_") the call node `i` is
        emitted with, None when it is emitted inline (libdevice, dd power chains, sqrt, fabs)."""
        n = self.node(i)
        if self.libm == "glibc-all" and n[1] in GL_FUNCTIONS and self.klass(i) in "PRCM":
            return "inflx_gl_"
        if self.klass(i) not in CR_CLASSES:
            return None
        if self.libm == "glibc" and n[1] in GL_FUNCTIONS:
            return "inflx_gl_"
        if self.libm == "cr" and n[1] in CR_FUNCTIONS:
            if n[1] == "pow" and self.dag.is_const(n[3]):
                # correctly rounded either way: the dd chains are ~100x cheaper
                e2 = 2.0 * float(self.dag.cval(n[3]))
                if e2.is_integer() and 1 <= abs(e2) <= 2 * MAX_FAST_POW:
                    return None
            return "inflx_cr_"
        return None

    def is_op(self, i: int) -> bool:
        return self.node(i)[0] in (
            "+", "-", "*", "/", "neg", "f", "rcp", "cmp", "and", "or", "not", "sel"
        )  # fmt: skip

    def nodes_of(self, classes: str, within=None) -> list[int]:
        src = self.all_nodes if within is None else within
        return [i for i in src if self.is_op(i) and self.klass(i) in classes]

    def flops(self, nodes) -> int:
        """Algorithmic flops of `nodes` by the SURVEY.md 8(d) rule (reciprocal pseudo-nodes are
        an implementation detail of the division and count as nothing)."""
        d = self.dag
        total = 0
        for i in nodes:
            n = self.node(i)
            k = n[0]
            if k in ("+", "-", "*", "/"):
                total += 1
            elif k == "f":
                if n[1] == "pow" and d.is_const(n[3]) and float(d.cval(n[3])).is_integer():
                    e = int(d.cval(n[3]))
                    total += _int_pow_mults(e) + (1 if e < 0 else 0)
                elif n[1] == "fabs":
                    pass
                else:
                    total += 1
        return total

    def stats(self) -> dict:
        g = self.grid_nodes
        ops = [i for i in g if self.is_op(i)]
        cnt = {c: len([i for i in ops if self.klass(i) == c]) for c in "PRCM"}
        per_point = [i for i in ops if self.klass(i) == "M"]
        return {
            "dag_ops": len([i for i in ops if self.node(i)[0] != "rcp"]),
            "class_ops": cnt,
            "flops_model": self.flops(ops),
            "flops_per_point_executed": self.flops(per_point),
            "divisions_per_point": len([i for i in per_point if self.node(i)[0] == "/"]),
            "reciprocals_per_point": len([i for i in per_point if self.node(i)[0] == "rcp"]),
            "n_p_frontier": len(self.p_frontier),
            "n_r_frontier": len(self.r_frontier),
            "n_row_slots": self.n_row_slots,
            "n_c_frontier": len(self.c_frontier),
            "n_c_live": len(self.c_live),
            "min_blocks": self.min_blocks,
            "transposed_store": self.transposed_store,
        }

    # -- emission ----------------------------------------------------------------------------
    def _ref(self, i: int, scope: dict[int, str]) -> str:
        """C expression naming node `i` inside a kernel whose already-bound values are `scope`."""
        if i in scope:
            return scope[i]
        n = self.node(i)
        if n[0] == "c":
            return _lit(n[1])
        if n[0] == "i":
            return _lit(float(n[1]))
        raise KeyError(f"node {i} {n} is not available in this scope")

    def _expr(self, i: int, scope: dict[int, str], spec: bool) -> str:
        """`spec`: branch-free speculative division / sqrt (per-point code of the grid kernels);
        otherwise the compiler's IEEE operators."""
        d = self.dag
        n = self.node(i)
        k = n[0]
        pol = "inflx_spec(bad)" if spec else "inflx_exact()"
        if k == "rcp":
            # a reciprocal read by a faster class carries the denominator's validity (NaN if not)
            hoisted = any(self.klass(u) != self.klass(i) for u in self.users.get(i, ()))
            fn = "inflx_rcp_checked" if hoisted else "inflx_rcp_s"
            return f"{fn}({self._ref(n[1], scope)})"
        if k == "/" and spec:
            rcp = self.rcp_of[n[2]]
            fn = "inflx_div_yh" if self.klass(rcp) != self.klass(i) else "inflx_div_y"
            y = self._ref(rcp, scope)
            if d.is_const(n[1]) and float(d.cval(n[1])) == 1.0:  # 1.0 / b: one DMUL less
                return f"{fn.replace('div', 'inv')}({self._ref(n[2], scope)}, {y}, bad)"
            return f"{fn}({self._ref(n[1], scope)}, {self._ref(n[2], scope)}, {y}, bad)"
        if k in ("+", "-", "*", "/"):
            return f"{self._ref(n[1], scope)} {k} {self._ref(n[2], scope)}"
        if k == "neg":
            return f"-{self._ref(n[1], scope)}"
        if k == "cmp":
            return f"(({self._ref(n[2], scope)} {n[1]} {self._ref(n[3], scope)}) ? 1.0 : 0.0)"
        if k in ("and", "or"):
            op = "&&" if k == "and" else "||"
            return (
                f"((({self._ref(n[1], scope)} != 0.0) {op} ({self._ref(n[2], scope)} != 0.0)) "
                "? 1.0 : 0.0)"
            )
        if k == "not":
            return f"(({self._ref(n[1], scope)} == 0.0) ? 1.0 : 0.0)"
        if k == "sel":
            # both arms are already evaluated (pure expressions); NaN / inf in the arm that is
            # not taken is discarded by the select exactly as the C conditional discards it
            return (
                f"(({self._ref(n[1], scope)} != 0.0) ? {self._ref(n[2], scope)} : "
                f"{self._ref(n[3], scope)})"
            )
        if k == "f":
            name = n[1]
            args = [self._ref(a, scope) for a in n[2:]]
            hoisted = self._hoisted_libm(i)
            if hoisted is not None:
                # evaluated once per parameter vector / grid row / grid column: afford the
                # reference's own libm (or the correctly rounded one), see LIBM_FLAVOURS
                if name == "pow" and hoisted == "inflx_gl_" and self.klass(i) == "M":
                    name = "pow_m"  # per point: main path inlined, the rest out of line
                return f"{hoisted}{name}({', '.join(args)})"
            if name == "pow" and d.is_const(n[3]):
                e = float(d.cval(n[3]))
                if e.is_integer() and 1 <= abs(e) <= MAX_FAST_POW:
                    e = int(e)
                    if e > 0:
                        return f"inflx_powi<{e}>({args[0]}, {pol})"
                    return f"inflx_powi_neg<{-e}>({args[0]}, {pol})"
                e2 = 2.0 * e
                if e2.is_integer() and abs(e2) <= 2 * MAX_FAST_POW:
                    e2 = int(e2)  # odd
                    if e2 > 0:
                        return f"inflx_powh<{(e2 - 1) // 2}>({args[0]}, {pol})"
                    return f"inflx_powh_neg<{(-e2 - 1) // 2}>({args[0]}, {pol})"
            if name == "sqrt" and spec:
                return f"inflx_sqrt_s({args[0]}, bad)"
            return f"{name}({', '.join(args)})"
        raise KeyError(f"cannot emit node {i}: {n}")

    def _block(self, nodes, scope, indent: str, spec: bool = False, lazy=None) -> str:
        """SSA statements for `nodes` (topological order); extends `scope` with their names.
        `lazy` maps not-yet-loaded nodes to their load expression: the load is emitted right
        before the first statement that uses the value (keeps live ranges short)."""
        out = []
        for i in nodes:
            if i in scope:
                continue
            if self.node(i)[0] == "rcp" and not spec:
                continue  # exact code divides with the IEEE operator and needs no reciprocal
            if lazy:
                for o in self.operands(i):
                    if o in lazy and o not in scope:
                        out.append(self._load(o, lazy, scope, indent))
            out.append(f"{indent}const double t{i} = {self._expr(i, scope, spec)};")
            scope[i] = f"t{i}"
        return "\n".join(out) + ("\n" if out else "")

    def _load(self, node: int, lazy: dict, scope: dict, indent: str) -> str:
        """Row-frontier values travel in pairs: one 128-bit warp-uniform load brings slot 2k and
        2k+1; the partner is bound too, so its own first use costs nothing."""
        slot = self.r_slot[node]
        pair = slot // 2
        names = {k: n for n, k in self.r_slot.items()}
        text = f"{indent}const double2 rp{pair} = rr[{pair}];\n"
        for half, member in ((2 * pair, "x"), (2 * pair + 1, "y")):
            n = names.get(half)
            if n is not None and n not in scope:
                scope[n] = f"rp{pair}.{member}"
        return text.rstrip("\n")

    def _leaf_scope(self, extra: dict[tuple, str]) -> dict[int, str]:
        """Names for leaves; `extra` maps ('x',0) etc. to C identifiers."""
        scope = {}
        for i in self.all_nodes:
            n = self.node(i)
            if n[0] in ("x", "p", "v1", "v2") and (n[0], n[1]) in extra:
                scope[i] = extra[(n[0], n[1])]
        return scope

    def cuda_source(self, model_name: str) -> str:
        with open(os.path.join(_CSRC, "inflx_device.cuh")) as fh:
            device_header = fh.read()
        if self.libm == "cr":
            with open(os.path.join(_CSRC, "inflx_crmath.cuh")) as fh:
                device_header += "\n" + fh.read()
        elif self.libm in ("glibc", "glibc-all"):
            with open(os.path.join(_CSRC, "inflx_glibc_tables.cuh")) as fh:
                tables = fh.read()
            with open(os.path.join(_CSRC, "inflx_glibcmath.cuh")) as fh:
                device_header += "\n" + fh.read().replace('#include "inflx_glibc_tables.cuh"', tables)
        npf, nrf = len(self.p_frontier), self.n_row_slots
        src = [f"#define INFLX_GROUP_MIN_BLOCKS {self.min_blocks}\n"]
        if self.libm == "glibc-all":  # the epilogue's atan / tan are the reference host's too
            src.append("#define INFLX_EXACT_ATAN_TAN 1\n")
        src.append(device_header)
        src.append(f'\n// ===== generated: model "{model_name}", group "{self.group}" =====\n')
        src.append(f"#define INFLX_NP {self.n_params}\n#define INFLX_NPF {npf}\n")
        src.append(f"#define INFLX_NRF {nrf}\n#define INFLX_PC_CAP {PC_CAPACITY}\n")
        src.append(f"#define INFLX_NCF {len(self.c_frontier)}\n")
        src.append(f"#define INFLX_SCALAR_XS {(self.n_params + 1) & ~1}\n")
        src.append("__constant__ double inflx_pc[INFLX_PC_CAP];\n")
        # feature marker the engine looks up: the grid kernels take (n_big, rpt_tail).  Its value is
        # the generator's advice: tail tiles of rpt / value rows; 0 = uniform tiles (a kernel bound
        # by the memory system gains nothing from a shorter drain and pays for the short tiles)
        tail_div = 0 if (self.group == "cmp" and self.transposed_store) else 4
        src.append(f'extern "C" __device__ const unsigned inflx_has_tail_tiles = {tail_div};\n\n')

        # ---- (1) parameter block: one thread per parameter vector ----
        scope = self._leaf_scope({("p", k): f"p[{k}]" for k in range(self.n_params)})
        body = self._block(self.nodes_of("P"), scope, "  ", spec=False)
        # reciprocals of P-class denominators are skipped by the exact block; emit the ones the
        # faster classes read
        for n in self.p_slot:
            if n not in scope and self.node(n)[0] == "rcp":
                body += f"  const double t{n} = {self._expr(n, scope, False)};\n"
                scope[n] = f"t{n}"
        stores = "".join(
            f"  pc[{k}] = {self._ref(n, scope)};\n" for n, k in self.p_slot.items()
        )
        src.append(
            "extern \"C\" __global__ void inflx_params(const double* __restrict__ p_all, "
            "double* __restrict__ pc_all, u32 n_vectors) {\n"
            "  const u32 s = blockIdx.x * blockDim.x + threadIdx.x;\n"
            "  if (s >= n_vectors) return;\n"
            "  const double* __restrict__ p = p_all + (u64)s * INFLX_NP;\n"
            "  double* __restrict__ pc = pc_all + (u64)s * INFLX_NPF;\n"
            "  (void)p; (void)pc;\n" + body + stores + "}\n\n"
        )

        # ---- (2) row block: one thread per (row, parameter vector) ----
        scope = {n: f"inflx_pc[pbase + {k}]" for n, k in self.p_slot.items()}
        scope.update(self._leaf_scope({("x", 0): "x0"}))
        body = self._block(self.nodes_of("R", self.grid_nodes), scope, "  ", spec=False)
        for n in self.r_slot:
            if n not in scope and self.node(n)[0] == "rcp":
                body += f"  const double t{n} = {self._expr(n, scope, False)};\n"
                scope[n] = f"t{n}"
        stores = "".join(
            f"  rr[{k}] = {self._ref(n, scope)};\n" for n, k in self.r_slot.items()
        )
        src.append(
            "extern \"C\" __global__ void inflx_rows(double* __restrict__ rc, double of0, double dx0, "
            "u64 row_begin, u32 n_rows) {\n"
            "  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;\n"
            "  if (i >= n_rows) return;\n"
            "  const u32 pbase = blockIdx.y * INFLX_NPF;\n"
            "  const double x0 = inflx_coord(row_begin + i, dx0, of0);\n"
            "  double* __restrict__ rr = rc + ((u64)blockIdx.y * n_rows + i) * INFLX_NRF;\n"
            "  (void)pbase; (void)x0; (void)rr;\n" + body + stores + "}\n\n"
        )

        # ---- (2a) fused prologue for ONE parameter vector: parameter block + row block in one launch.
        # The parameters arrive BY VALUE in the kernel's argument buffer (no H2D copy), every thread
        # evaluates the (cheap) parameter block itself and then its row; thread 0 also writes the
        # P-frontier values out for the copy into the grid kernel's __constant__ bank.  Replaces
        # H2D + inflx_params + inflx_rows on a call's first row chunk: 5 dependent operations in
        # front of the grid kernel become 3 (the ~47 us serial prologue of round 1 is what a
        # 1 ms step on 8 GPUs loses most).  Same operations -> same bits.
        scope = self._leaf_scope({("p", k): f"pv.v[{k}]" for k in range(self.n_params)})
        scope.update(self._leaf_scope({("x", 0): "x0"}))
        body_p = self._block(self.nodes_of("P"), scope, "  ", spec=False)
        for n in self.p_slot:
            if n not in scope and self.node(n)[0] == "rcp":
                body_p += f"  const double t{n} = {self._expr(n, scope, False)};\n"
                scope[n] = f"t{n}"
        stores_p = "".join(
            f"    pc_out[{k}] = {self._ref(n, scope)};\n" for n, k in self.p_slot.items()
        )
        body_r = self._block(self.nodes_of("R", self.grid_nodes), scope, "  ", spec=False)
        for n in self.r_slot:
            if n not in scope and self.node(n)[0] == "rcp":
                body_r += f"  const double t{n} = {self._expr(n, scope, False)};\n"
                scope[n] = f"t{n}"
        stores_r = "".join(
            f"  rr[{k}] = {self._ref(n, scope)};\n" for n, k in self.r_slot.items()
        )
        src.append(
            f"struct inflx_pvec {{ double v[{max(self.n_params, 1)}]; }};\n"
            "extern \"C\" __global__ void inflx_prologue(const inflx_pvec pv, "
            "double* __restrict__ pc_out, double* __restrict__ rc, double of0, double dx0, "
            "u64 row_begin, u32 n_rows) {\n"
            "  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;\n"
            "  const double x0 = inflx_coord(row_begin + (i < n_rows ? i : 0u), dx0, of0);\n"
            "  (void)x0; (void)pv;\n" + body_p
            + "  if (i == 0) {\n" + stores_p + "  }\n"
            "  if (i >= n_rows) return;\n"
            "  double* __restrict__ rr = rc + (u64)i * INFLX_NRF;\n  (void)rr;\n"
            + body_r + stores_r + "}\n\n"
        )

        # ---- (2b) column block as a pre-pass: one thread per (column, parameter vector) ----
        if self.cols_prepass:
            scope = {n: f"inflx_pc[pbase + {k}]" for n, k in self.p_slot.items()}
            scope.update(self._leaf_scope({("x", 1): "x1"}))
            body = self._block(self.nodes_of("C", self.grid_nodes), scope, "  ", spec=False)
            for n in self.c_slot:
                if n not in scope and self.node(n)[0] == "rcp":
                    body += f"  const double t{n} = {self._expr(n, scope, False)};\n"
                    scope[n] = f"t{n}"
            stores = "".join(
                f"  cc[((u64)blockIdx.y * INFLX_NCF + {k}) * n1 + col] = {self._ref(n, scope)};\n"
                for n, k in self.c_slot.items()
            )
            src.append(
                "extern \"C\" __global__ void inflx_cols(double* __restrict__ cc, double of1, "
                "double dx1, u32 n1) {\n"
                "  const u32 col = blockIdx.x * blockDim.x + threadIdx.x;\n"
                "  if (col >= n1) return;\n"
                "  const u32 pbase = blockIdx.y * INFLX_NPF;\n"
                "  const double x1 = inflx_coord(col, dx1, of1);\n"
                "  (void)pbase; (void)x1;\n" + body + stores + "}\n\n"
            )

        # ---- (3) slow path + grid kernels: thread = column, walks INFLX_RPT rows ----
        src.append(self._slow_function())
        for op in self.grid_ops:
            for sweep in (False, True):
                src.append(self._grid_kernel(op, sweep))
        # ---- (4) point kernels (on-trajectory / scalar entry points) ----
        for op in self.point_ops:
            src.append(self._point_kernel(op))
            if op in SCALAR_OPS:
                src.append(self._scalar_kernel(op))
        return "".join(src)

    def _epilogue(self, op: str, val, point: str, indent: str, spec: bool) -> str:
        """Statement(s) writing the result of `op` for the point with flat index `point`."""
        s, b = ("_s", ", bad") if spec else ("", "")
        if op == "complete_analysis":
            if spec and self._v10_is_plus_zero():
                return (
                    f"{indent}o6 = inflx_op_complete_v10z_s({val('V')}, {val('v00')}, "
                    f"{val('v11')}, {val('g2')}, bad);\n"
                )
            return (
                f"{indent}o6 = inflx_op_complete{s}({val('V')}, {val('v00')}, "
                f"{val('v10')}, {val('v11')}, {val('g2')}{b});\n"
            )
        if op == "consistency_only" and spec and self._v10_is_plus_zero():
            return f"{indent}o1 = inflx_op_consistency_v10z_s();\n"
        if op == "consistency_rapidturn_only" and spec and self._v10_is_plus_zero():
            return (
                f"{indent}o1 = inflx_op_rapidturn_v10z_s({val('V')}, {val('v00')}, "
                f"{val('v11')}, bad);\n"
            )
        if op == "consistency_only":
            return (
                f"{indent}o1 = inflx_op_consistency{s}({val('V')}, {val('v00')}, "
                f"{val('v10')}, {val('v11')}{b});\n"
            )
        if op == "consistency_rapidturn_only":
            return (
                f"{indent}o1 = inflx_op_rapidturn{s}({val('V')}, {val('v00')}, "
                f"{val('v10')}, {val('v11')}{b});\n"
            )
        if op == "epsilon_v_only":
            return f"{indent}o1 = inflx_op_epsilon_v{s}({val('V')}, {val('g2')}{b});\n"
        if op == "flag_quantum_dif":
            return f"{indent}o1 = (double)inflx_op_flag({val('b0')}, {val('b1')}, aux);\n"
        if op == "potential":
            return f"{indent}o1 = {val('V')};\n"
        if op == "hesse":
            return "".join(
                f"{indent}o4[{c}] = {val(nm)};\n"
                for c, nm in enumerate(("v00", "v01", "v10", "v11"))
            )
        raise KeyError(op)

    def _v10_is_plus_zero(self) -> bool:
        """v10 (V_wv) is the compile-time constant +0.0 and no other root is a constant: the
        complete_analysis epilogue has a closed special form (inflx_op_complete_v10z_s)."""
        r = self.grid_roots
        if "v10" not in r or not self.dag.is_const(r["v10"]):
            return False
        z = float(self.dag.cval(r["v10"]))
        if z != 0.0 or math.copysign(1.0, z) < 0:
            return False
        return not any(self.klass(n) == "K" for nm, n in r.items() if nm != "v10")

    def _store(self, op: str, point: str, indent: str) -> str:
        if op == "complete_analysis":
            return f"{indent}inflx_store6(out, {point}, o6);\n"
        if op == "flag_quantum_dif":
            return f"{indent}reinterpret_cast<unsigned char*>(out)[{point}] = (unsigned char)(o1 != 0.0);\n"
        if op == "hesse":
            # (2,2,N0,N1) component-major output (reference src/hesse_bindings.rs:150-192)
            return "".join(
                f"{indent}out[{c}ull * comp_stride + {point}] = o4[{c}];\n" for c in range(4)
            )
        return f"{indent}out[{point}] = o1;\n"

    def _root_order(self) -> list[str]:
        return list(self.grid_roots)

    def _slow_function(self) -> str:
        """Exact (IEEE-operator) recomputation of the group's root values at one grid point; run
        only for points whose speculative division / sqrt left the validated range."""
        scope = {n: f"inflx_pc[pbase + {k}]" for n, k in self.p_slot.items()}
        scope.update(self._leaf_scope({("x", 1): "x1"}))
        lazy = {n: f"__ldg(rr + {k})" for n, k in self.r_slot.items()}
        body = self._block(self.nodes_of("CM", self.grid_nodes), scope, "  ", False, lazy)
        outs = ""
        for k, nm in enumerate(self._root_order()):
            r = self.grid_roots[nm]
            if r in lazy and r not in scope:
                outs += self._load(r, lazy, scope, "  ") + "\n"
            outs += f"  roots[{k}] = {self._ref(r, scope)};\n"
        return (
            "__device__ __noinline__ void inflx_slow_roots(const double2* __restrict__ rr, double x1, "
            "u32 pbase, double* __restrict__ roots) {\n  (void)rr; (void)x1; (void)pbase;\n"
            + body + outs + "}\n\n"
        )

    def _grid_kernel(self, op: str, sweep: bool) -> str:
        name = f"inflx_grid_{op}" + ("_sweep" if sweep else "")
        pbase = "pbase + " if sweep else ""
        scope = {n: f"inflx_pc[{pbase}{k}]" for n, k in self.p_slot.items()}
        scope.update(self._leaf_scope({("x", 1): "x1"}))
        if self.cols_prepass:
            # column-frontier values come from the inflx_cols pre-pass: coalesced loads
            col_block = "  const u32 ccol = active ? col : 0u;\n"
            for n, k in self.c_slot.items():
                col_block += (
                    f"  const double t{n} = __ldg(cc + ((u64)s * INFLX_NCF + {k}) * n1 + ccol);\n"
                )
                scope[n] = f"t{n}"
        else:
            col_block = self._block(self.nodes_of("C", self.grid_nodes), scope, "  ", spec=True)
            col_block = col_block.replace(", bad)", ", bad_c)").replace("(bad)", "(bad_c)")
        lazy = {n: f"__ldg(rr + {k})" for n, k in self.r_slot.items()}
        mixed = self._block(self.nodes_of("M", self.grid_nodes), scope, "    ", True, lazy)
        root_loads = ""
        for nm, r in self.grid_roots.items():  # roots that are plain row-frontier values
            if r in lazy and r not in scope:
                root_loads += self._load(r, lazy, scope, "    ") + "\n"

        def val(rname: str) -> str:
            return self._ref(self.grid_roots[rname], scope)

        order = self._root_order()

        def slow_val(rname: str) -> str:
            return f"roots[{order.index(rname)}]"

        decl = {"complete_analysis": "inflx_six o6;", "hesse": "double o4[4];"}.get(op, "double o1;")
        transposed = op == "complete_analysis" and self.transposed_store
        # a root that is a compile-time constant (hyperinflation: v10 == 0) would send EVERY point
        # of the speculative epilogue to the slow path (x/0); use the IEEE epilogue directly then
        spec_epi = not any(self.klass(r) == "K" for r in self.grid_roots.values()) or (
            op in ("complete_analysis", "consistency_only", "consistency_rapidturn_only")
            and self._v10_is_plus_zero()
        )
        return (
            f"extern \"C\" __global__ void __launch_bounds__(INFLX_BLOCK, INFLX_MIN_BLOCKS) {name}("
            "double* __restrict__ out, const double* __restrict__ rc, double of1, double dx1, "
            "u32 n1, u32 n_rows, u64 comp_stride, double aux, u32 rpt, "
            "const double* __restrict__ cc, u32 n_big, u32 rpt_tail) {\n"
            "  const u32 col = blockIdx.x * INFLX_BLOCK + threadIdx.x;\n"
            + (
                "  const u32 s = blockIdx.z;\n  const u32 pbase = s * INFLX_NPF;\n"
                if sweep
                else "  const u32 s = 0;\n  const u32 pbase = 0;\n"
            )
            # rows per CTA: chosen per launch by the engine (<= INFLX_RPT, which sizes the smem).
            # Two tile heights: the first n_big row tiles walk `rpt` rows, the rest `rpt_tail`
            # (<= rpt) - CTAs are dispatched in blockIdx order, so the launch ENDS on short CTAs
            # and the last wave drains in a fraction of a full tile's duration.
            + "  const bool tail = blockIdx.y >= n_big;\n"
            "  const u32 r0 = tail ? n_big * rpt + (blockIdx.y - n_big) * rpt_tail : blockIdx.y * rpt;\n"
            "  const u32 rows_here = min(tail ? rpt_tail : rpt, n_rows - r0);\n"
            # the CTA's rows of the row-frontier array: one cooperative, coalesced 128-bit copy
            # into shared memory, overlapped with the column block; per-point reads are then
            # conflict-free LDS.128 broadcasts instead of exposed L2 round trips
            "#if INFLX_NRF > 0\n"
            "  __shared__ double2 rsm[INFLX_RPT * (INFLX_NRF / 2)];\n"
            "  {\n"
            "    const double2* __restrict__ src = reinterpret_cast<const double2*>(\n"
            "        rc + ((u64)s * n_rows + r0) * INFLX_NRF);\n"
            "    for (u32 k = threadIdx.x; k < rows_here * (INFLX_NRF / 2); k += INFLX_BLOCK)\n"
            "      rsm[k] = __ldg(src + k);\n"
            "  }\n"
            "#endif\n"
            + ("  __shared__ double2 inflx_st[(INFLX_BLOCK + 31) / 32][96];\n" if transposed else "")
            + "  const bool active = col < n1;\n"
            "  const double x1 = inflx_coord(active ? col : 0u, dx1, of1);\n"
            "  inflx_chk bad_c;\n"
            "  (void)x1; (void)aux; (void)comp_stride; (void)rc; (void)pbase; (void)cc;\n"
            + col_block
            + "#if INFLX_NRF > 0\n  __syncthreads();\n#endif\n"
            # transposed stores are a warp-wide operation: lanes beyond the grid's last column keep
            # computing (on column 0) and are masked out of the store instead of leaving
            + ("  const u32 warp_col0 = col - (threadIdx.x & 31u);\n"
               "  const u32 n_valid = warp_col0 < n1 ? min(32u, n1 - warp_col0) : 0u;\n"
               if transposed else "  if (!active) return;\n")
            + "#pragma unroll 1\n"
            "  for (u32 j = 0; j < rows_here; ++j) {\n"
            "    const u64 rowid = (u64)s * n_rows + r0 + j;\n"
            "#if INFLX_NRF > 0\n"
            "    const double2* __restrict__ rr = rsm + j * (INFLX_NRF / 2);\n"
            "#else\n"
            "    const double2* __restrict__ rr = nullptr;\n"
            "#endif\n"
            "    const u64 point = rowid * n1 + col;\n"
            "    inflx_chk bad = bad_c;\n"
            f"    {decl}\n"
            "    (void)rr;\n"
            + mixed
            + root_loads
            + self._epilogue(op, val, "point", "    ", spec_epi)
            # the speculative result is stored as soon as it exists (its registers are free before
            # the validity flag is final) and overwritten by the rare recomputation;
            # -DINFLX_LATE_STORE: one store after the flag is known (round 1)
            + ("" if transposed else "#ifndef INFLX_LATE_STORE\n" + self._store(op, "point", "    ") + "#endif\n")
            + "    if (bad.any()) {  // rare: redo this point with the IEEE operators\n"
            f"      double roots[{len(order)}];\n"
            "      inflx_slow_roots(rr, x1, pbase, roots);\n"
            + self._epilogue(op, slow_val, "point", "      ", False)
            + ("" if transposed else "#ifndef INFLX_LATE_STORE\n" + self._store(op, "point", "      ") + "#endif\n")
            + "    }\n"
            + (
                "    inflx_store6_warp(out, rowid * n1 + warp_col0, n_valid, o6, "
                "inflx_st[threadIdx.x >> 5]);\n"
                if transposed
                else "#ifdef INFLX_LATE_STORE\n" + self._store(op, "point", "    ") + "#endif\n"
            )
            + "  }\n}\n\n"
        )

    def _point_kernel(self, op: str) -> str:
        """One thread per explicit field-space point (reference src/anguelova.rs:633-977 and the
        scalar entry points src/lib.rs:309-339, 384-419): coordinates are loaded, not generated."""
        scope = {n: f"inflx_pc[{k}]" for n, k in self.p_slot.items()}
        scope.update(self._leaf_scope({("x", 0): "x0", ("x", 1): "x1"}))
        roots = self.point_roots if op == "basis" else self.grid_roots
        want = [r for nm, r in roots.items() if nm != "ip"]
        nodes = [i for i in self.dag.reachable(want) if self.is_op(i) and self.klass(i) in "RCM"]
        body = self._block(nodes, scope, "  ", spec=False)

        def val(rname: str) -> str:
            return self._ref(roots[rname], scope)

        pre = ""
        if op == "hesse":
            epi = "  double o4[4];\n" + self._epilogue(op, val, "k", "  ", False)
            epi += "".join(f"  out[k * 4 + {c}] = o4[{c}];\n" for c in range(4))
        elif op == "basis":
            # v, w1 and the three metric inner products (reference src/lib.rs:142-203)
            pre = self._inner_function()
            epi = (
                f"  const double b0 = {val('b0')}, b1 = {val('b1')}, w0 = {val('w0')}, w1 = {val('w1')};\n"
                "  out[k * 7 + 0] = b0; out[k * 7 + 1] = b1; out[k * 7 + 2] = w0; out[k * 7 + 3] = w1;\n"
                "  out[k * 7 + 4] = inflx_inner(x0, x1, b0, b1, b0, b1);\n"
                "  out[k * 7 + 5] = inflx_inner(x0, x1, b0, b1, w0, w1);\n"
                "  out[k * 7 + 6] = inflx_inner(x0, x1, w0, w1, w0, w1);\n"
            )
        else:
            decl = "inflx_six o6;" if op == "complete_analysis" else "double o1;"
            epi = f"  {decl}\n" + self._epilogue(op, val, "k", "  ", False) + self._store(op, "k", "  ")
        return (
            pre
            + f"extern \"C\" __global__ void inflx_points_{op}(double* __restrict__ out, "
            "const double* __restrict__ xs, u64 n, double aux) {\n"
            "  const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;\n"
            "  if (k >= n) return;\n"
            "  const double2 xx = reinterpret_cast<const double2*>(xs)[k];\n"
            "  const double x0 = xx.x, x1 = xx.y;\n"
            "  (void)x0; (void)x1; (void)aux;\n" + body + epi + "}\n\n"
        )

    def _scalar_kernel(self, op: str) -> str:
        """The scalar entry points `potential(x, p)` / `hesse(x, p)` (reference src/lib.rs:309-339,
        384-419) as ONE launch: every class of the group - parameter block included - evaluated
        inline by the thread, parameters and coordinates read from, and the result written to,
        mapped page-locked host memory.  The general path costs H2D + inflx_params + DtoD into
        __constant__ + H2D + inflx_points_* + D2H per call; this one a launch and a stream
        synchronise.  Same operations, same libm flavour per node class as the two-kernel path, so
        the values are bit-identical to inflx_points_<op>."""
        scope = self._leaf_scope(
            {("p", k): f"p[{k}]" for k in range(self.n_params)} | {("x", 0): "x0", ("x", 1): "x1"}
        )
        roots = self.grid_roots
        nodes = [
            i for i in self.dag.reachable(list(roots.values()))
            if self.is_op(i) and self.klass(i) in "PRCM"
        ]
        body = self._block(nodes, scope, "  ", spec=False)

        def val(rname: str) -> str:
            return self._ref(roots[rname], scope)

        if op == "hesse":
            epi = "  double o4[4];\n" + self._epilogue(op, val, "k", "  ", False)
            epi += "".join(f"  out[k * 4 + {c}] = o4[{c}];\n" for c in range(4))
        else:
            epi = "  double o1;\n" + self._epilogue(op, val, "k", "  ", False) + "  out[k] = o1;\n"
        return (
            f"extern \"C\" __global__ void inflx_scalar_{op}(double* __restrict__ out, "
            "const double* __restrict__ in, u64 n) {\n"
            "  const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;\n"
            "  if (k >= n) return;\n"
            "  const double* __restrict__ p = in;\n"
            "  const double x0 = in[INFLX_SCALAR_XS + 2 * k], x1 = in[INFLX_SCALAR_XS + 2 * k + 1];\n"
            "  (void)p; (void)x0; (void)x1;\n" + body + epi + "}\n\n"
        )

    def _inner_function(self) -> str:
        """`inner_prod` (reference compiler.py:445-472) as a device function of the two vectors."""
        scope = {n: f"inflx_pc[{k}]" for n, k in self.p_slot.items()}
        scope.update(
            self._leaf_scope({
                ("x", 0): "x0", ("x", 1): "x1", ("v1", 0): "a0", ("v1", 1): "a1",
                ("v2", 0): "c0", ("v2", 1): "c1",
            })  # fmt: skip
        )
        root = self.point_roots["ip"]
        nodes = [
            i for i in self.dag.reachable([root]) if self.is_op(i) and self.klass(i) in "RCMV"
        ]
        body = self._block(nodes, scope, "  ", spec=False)
        return (
            "__device__ __noinline__ double inflx_inner(double x0, double x1, double a0, double a1, "
            "double c0, double c1) {\n  (void)x0; (void)x1; (void)a0; (void)a1; (void)c0; (void)c1;\n"
            + body
            + f"  return {self._ref(root, scope)};\n}}\n\n"
        )


class ModelProgram:
    """All groups of one model + the metadata the artefact header carries."""

    def __init__(self, unit: ParsedUnit, libm: str = "glibc", cols: str = "auto",
                 store: str = "auto"):
        self.libm = libm
        if unit.dim != 2:
            raise Exception(
                f"the CUDA back-end evaluates 2-field models (the model has {unit.dim} fields)"
            )
        self.unit = unit
        self.roots = ModelRoots(unit)
        self.groups = {
            g: GroupProgram(unit.dag, self.roots, g, unit.n_parameters or 0, libm, cols, store)
            for g in GROUPS
        }

    def flops_per_point(self, op: str) -> int:
        """F(model, op) of SURVEY.md 8(d): joint-CSE DAG of the functions `op` reads + epilogue."""
        for g, (_, _, grid_ops, point_ops) in GROUPS.items():
            if op in grid_ops or op in point_ops:
                gp = self.groups[g]
                ops = [i for i in gp.grid_nodes if gp.is_op(i)]
                return gp.flops(ops) + EPILOGUE_FLOPS[op]
        raise KeyError(op)

    def metadata(self) -> dict:
        meta = {}
        for g, gp in self.groups.items():
            st = gp.stats()
            st["grid_ops"] = list(gp.grid_ops)
            st["point_ops"] = list(gp.point_ops)
            meta[g] = st
        flops = {}
        for g, (_, _, grid_ops, point_ops) in GROUPS.items():
            for op in set(grid_ops) | set(point_ops):
                if op != "basis":
                    flops[op] = self.flops_per_point(op)
        return {"groups": meta, "flops_per_point": flops, "libm": self.libm}
