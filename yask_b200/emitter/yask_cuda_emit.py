#!/usr/bin/env python
"""CUDA emitter for YASK stencil solutions (build-time tool).

Pipeline:  DSL (src/stencils/*.cpp, unchanged)  ->  the reference's own compiler FRONT-END
(`yask_compiler.exe`: parsing, CSE/combination, dependency analysis, part/stage formation, halo and
step-allocation analysis; /root/reference/src/compiler/lib/Solution.cpp:127-160)  ->  this emitter,
which replaces the reference's AVX/C++ back-end (`Cpp.cpp`, `CppIntrin.cpp`, `YaskKernel.cpp`).

The front-end is used as a black box through the file it already writes: we ask it for its C++ target
and read (a) the per-var metadata block (alloc_t, halos, L1 norms -- what the generated context ctor
encodes, YaskKernel.cpp:730-) and (b) the `calc_scalar()` bodies, which list every part's expression tree
as a sequence of single-assignment statements in evaluation order with 16-digit constants
(Cpp.cpp:39-53).  The vector path the reference actually runs evaluates the SAME trees with the constants
rounded to the element type, every op in the element type -- that is the semantics we emit.

Outputs (committed; nothing at run time needs the reference):
  yask_b200/csrc/gen/<name>.gen.cuh   CUDA kernels (one per part) + the StencilSpec table
  oracle/gen/<name>.gen.h             plain-C restatement of the same statements (TEST oracle)
  yask_b200/csrc/gen/<name>.json      the parsed IR (tests use it for var names / halos)

Covered: sub-domain (IF_DOMAIN) and step (IF_STEP) conditions, scratch vars and scratch-part chains, the DSL's math
functions, misc dims (up to two per var), 1-D/2-D/3-D solutions, reverse-time solutions.  Refused with a message (never
silently dropped): more than three domain dims, more than two misc dims per var, non-constant misc indices.

usage: python -m yask_b200.emitter.yask_cuda_emit --stencil awp_elastic --elem-bytes 4 [--radius R] [--name NAME]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
# The reference's stencil compiler, built out of tree from the unmodified sources by oracle/build_ref.sh into
# oracle/_ref/ship/refc (the emitter's outputs are committed, nothing at run time needs it).
REFC = os.path.join(ROOT, "oracle", "_ref", "ship", "refc")
COMPILER = os.path.join(REFC, "bin", "yask_compiler.exe")
COMPILER_LIB = os.path.join(REFC, "lib")


class EmitError(RuntimeError):
    pass


def c_ident(name: str) -> str:
    """C identifier for a solution name ("3axis" -> "s3axis")."""
    i = re.sub(r"\W", "_", name)
    return ("s" + i) if i[0].isdigit() else i


# ----------------------------------------------------------------------------------------------------
# front-end: run the reference compiler and parse its output
# ----------------------------------------------------------------------------------------------------
def run_frontend(stencil: str, elem_bytes: int, radius: int | None) -> str:
    if not os.path.exists(COMPILER):
        raise EmitError(f"{COMPILER} missing: run oracle/build_ref.sh first (needs the reference's sources)")
    with tempfile.TemporaryDirectory() as d:
        out = os.path.join(d, "gen.hpp")
        cmd = [COMPILER, "-stencil", stencil, "-target", "avx512", "-elem-bytes", str(elem_bytes), "-p", out]
        if radius:
            cmd += ["-radius", str(radius)]
        env = dict(os.environ, LD_LIBRARY_PATH=COMPILER_LIB + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
        r = subprocess.run(cmd, env=env, capture_output=True, text=True)
        if r.returncode != 0 or not os.path.exists(out):
            raise EmitError("reference compiler failed:\n" + r.stdout[-2000:] + r.stderr[-2000:])
        return open(out).read()


_NUM = r"[-+]?(?:\d+\.\d*(?:[eE][-+]?\d+)?|\.\d+(?:[eE][-+]?\d+)?|\d+(?:[eE][-+]?\d+)?)"


def parse_index(tok: str, dims: list[str]):
    """'x' | '(x - 1)' | '(t + 1)' | '3' -> (dim or None, offset)"""
    tok = tok.strip()
    m = re.fullmatch(r"\(?\s*([A-Za-z_]\w*)\s*(?:([-+])\s*(\d+))?\s*\)?", tok)
    if m:
        off = int(m.group(3)) if m.group(3) else 0
        return m.group(1), (-off if m.group(2) == "-" else off)
    if re.fullmatch(r"-?\d+", tok):
        return None, int(tok)
    raise EmitError(f"unsupported index expression '{tok}'")


def parse_domain_cond(text: str, dd: list[str]) -> dict:
    """Sub-domain condition of a part (IF_DOMAIN in the DSL; printed by the reference as a C expression over the
    GLOBAL domain indices with FIRST_INDEX(d)/LAST_INDEX(d) for the overall problem bounds).
    Returns {"expr": neutral C text using G(i), GF(i), GL(i); "bounds": per-dim [lo, hi] affine bounds when the
    expression is a conjunction of simple comparisons (used to shrink the launch box), else None}."""
    t = text.strip()
    if len(dd) > 3:
        raise EmitError("more than 3 domain dims are not supported")
    sh = 3 - len(dd)          # kernel slot of domain dim i is i + sh
    for i, d in enumerate(dd):
        t = re.sub(rf"FIRST_INDEX\(\s*{d}\s*\)", f"GF({i + sh})", t)
        t = re.sub(rf"LAST_INDEX\(\s*{d}\s*\)", f"GL({i + sh})", t)
    for i, d in enumerate(dd):
        t = re.sub(rf"(?<!\w){d}(?!\w)", f"G({i + sh})", t)
    left = re.sub(r"G[FL]?\(\d\)|\d+|[-+*/%()<>=!&| ]", "", t)
    if left:
        raise EmitError(f"unsupported token(s) '{left}' in sub-domain condition '{text}'")
    # bounds: conjunction of  G(i) OP (affine in GF/GL(i) and integers)
    bounds = {}
    ok = True

    def strip_parens(x):
        x = x.strip()
        while x.startswith("(") and x.endswith(")"):
            depth, good = 0, True
            for k, ch in enumerate(x):
                depth += ch == "("
                depth -= ch == ")"
                if depth == 0 and k < len(x) - 1:
                    good = False
                    break
            if not good:
                break
            x = x[1:-1].strip()
        return x

    def split_top(x, sep):
        parts, depth, cur, k = [], 0, "", 0
        while k < len(x):
            ch = x[k]
            depth += ch == "("
            depth -= ch == ")"
            if depth == 0 and x.startswith(sep, k):
                parts.append(cur)
                cur = ""
                k += len(sep)
                continue
            cur += ch
            k += 1
        parts.append(cur)
        return parts

    for term in split_top(strip_parens(t), "&&"):
        term = strip_parens(term)
        m = re.fullmatch(r"G\((\d)\)\s*(==|<=|>=|<|>)\s*(.+)", term)
        if not m or "||" in term:
            ok = False
            break
        i, op, rhs = int(m.group(1)), m.group(2), m.group(3)
        # evaluate rhs symbolically as base + off with base in {GF(i), GL(i), none}
        probe = {}
        for base in ("GF", "GL"):
            if re.search(rf"{base}\((?!{i}\))", rhs):
                ok = False
        if not ok:
            break
        try:
            v0 = eval(rhs.replace(f"GF({i})", "0").replace(f"GL({i})", "0"), {"__builtins__": {}})
            vf = eval(rhs.replace(f"GF({i})", "1").replace(f"GL({i})", "0"), {"__builtins__": {}})
            vl = eval(rhs.replace(f"GF({i})", "0").replace(f"GL({i})", "1"), {"__builtins__": {}})
        except Exception:
            ok = False
            break
        cf, cl = vf - v0, vl - v0
        if (cf, cl) not in ((0, 0), (1, 0), (0, 1)):
            ok = False
            break
        base = "GF" if cf else ("GL" if cl else "0")
        lo, hi = bounds.get(i, [None, None])
        b = [base, int(v0)]
        if op == "==":
            lo, hi = b, b
        elif op == "<=":
            hi = b
        elif op == "<":
            hi = [base, int(v0) - 1]
        elif op == ">=":
            lo = b
        elif op == ">":
            lo = [base, int(v0) + 1]
        bounds[i] = [lo, hi]
    return {"expr": t, "bounds": {str(k): v for k, v in bounds.items()} if ok else None, "text": text.strip()}


# DSL math functions (/root/reference/src/kernel/lib/realv.hpp:713-726) -> number of arguments
MATH_FUNCS = {"sqrt": 1, "cbrt": 1, "fabs": 1, "erf": 1, "exp": 1, "log": 1, "sin": 1, "cos": 1, "atan": 1,
              "pow": 2, "min": 2, "max": 2}


class Parser:
    """Tiny recursive-descent parser for the RHS of generated statements: + - * / with C precedence and
    left associativity, parentheses, unary minus, numeric literals, expr_temp refs and read placeholders."""

    def __init__(self, text: str):
        self.toks = re.findall(r"@\d+|(?:arg\d+|res|expr)_temp\d+|yask_\w+|" + r"\d+\.\d*(?:[eE][-+]?\d+)?|\d+(?:[eE][-+]?\d+)?" + r"|[-+*/(),]", text)
        joined = "".join(self.toks)
        if joined != re.sub(r"\s+", "", text):
            raise EmitError(f"unsupported construct in expression: '{text}'")
        self.i = 0

    def peek(self):
        return self.toks[self.i] if self.i < len(self.toks) else None

    def next(self):
        t = self.peek()
        self.i += 1
        return t

    def parse(self):
        e = self.expr()
        if self.peek() is not None:
            raise EmitError("trailing tokens in expression")
        return e

    def expr(self):
        e = self.term()
        while self.peek() in ("+", "-"):
            op = self.next()
            e = ("add" if op == "+" else "sub", e, self.term())
        return e

    def term(self):
        e = self.unary()
        while self.peek() in ("*", "/"):
            op = self.next()
            e = ("mul" if op == "*" else "div", e, self.unary())
        return e

    def unary(self):
        if self.peek() == "-":
            self.next()
            nxt = self.peek()
            if nxt and re.fullmatch(r"\d.*", nxt):   # negative literal
                return ("const", "-" + self.next())
            return ("neg", self.unary())
        if self.peek() == "+":
            self.next()
        return self.atom()

    def atom(self):
        t = self.next()
        if t is None:
            raise EmitError("unexpected end of expression")
        if t == "(":
            e = self.expr()
            if self.next() != ")":
                raise EmitError("missing ')'")
            return e
        if t.startswith("@"):
            return ("read", int(t[1:]))
        m = re.fullmatch(r"(expr|res|arg(\d+))_temp(\d+)", t)
        if m:
            return ("tmp", {"expr": "e", "res": "r"}.get(m.group(1), f"a{m.group(2)}_") + m.group(3))
        if t.startswith("yask_"):
            fn = t[len("yask_"):]
            if fn not in MATH_FUNCS:
                raise EmitError(f"unsupported math function '{t}'")
            if self.next() != "(":
                raise EmitError(f"'(' expected after {t}")
            args = [self.expr()]
            while self.peek() == ",":
                self.next()
                args.append(self.expr())
            if self.next() != ")":
                raise EmitError("missing ')'")
            if len(args) != MATH_FUNCS[fn]:
                raise EmitError(f"{t}: {len(args)} argument(s)")
            return ("call", fn, args)
        return ("const", t)


def parse_generated(text: str, name: str) -> dict:
    ir: dict = {"name": name, "vars": [], "stages": []}
    # ---- element size, dims --------------------------------------------------------------------------
    m = re.search(r"#define REAL_BYTES \((\d+)\)", text) or re.search(r"REAL_BYTES\s+\(?(\d+)\)?", text)
    ir["elem_bytes"] = int(m.group(1)) if m else None
    # ---- vars -----------------------------------------------------------------------------------------
    for m in re.finditer(r"// The (?:(\d+)-D var|scalar value) '(\w+)', which is\s+(updated by one or more equations|not updated by any equation|a scratch variable)[^\n]*\n"
                         r"(?:\s*// Dimensions in parameter \(declaration\) order: ([^\n]*)\n)?", text):
        vname = m.group(2)
        dims = re.findall(r"'(\w+)'\(#\d+\)", m.group(4) or "")
        if any(v["name"] == vname for v in ir["vars"]):
            continue
        ir["vars"].append({"name": vname, "dims": dims, "is_output": m.group(3).startswith("updated"),
                           "scratch": m.group(3).startswith("a scratch")})
    ir["vars"].sort(key=lambda v: v["scratch"])      # scratch vars last (stable): they are engine-internal storage
    if not ir["vars"]:
        raise EmitError("no vars found in the generated file")
    # domain dims: the front-end's own list ("#define DOMAIN_DIM_IDX_<d> <i>"); step dim: the first dim of an updated var
    dd = [d for d, _ in sorted(re.findall(r"#define DOMAIN_DIM_IDX_(\w+) (\d+)", text), key=lambda kv: int(kv[1]))]
    step_dim = None
    for v in ir["vars"]:
        if v["is_output"] and v["dims"] and v["dims"][0] not in dd:
            step_dim = v["dims"][0]
    if not dd:
        raise EmitError("no domain dims found in the generated file")
    ir["step_dim"], ir["domain_dims"] = step_dim, dd
    if len(dd) > 3:
        raise EmitError(f"{len(dd)} domain dims: more than 3 are not supported")
    for v in ir["vars"]:
        n = v["name"]
        m = re.search(rf"const idx_t {n}_alloc_{step_dim} = (\d+);", text)
        v["alloc_t"] = int(m.group(1)) if m else 1
        m = re.search(rf"const int {n}_l1_norm = (\d+);", text)
        v["l1_norm"] = int(m.group(1)) if m else 0
        v["halo"] = {}
        for d in v["dims"]:
            if d == step_dim:
                continue
            if d not in dd:
                continue      # misc dim: its index range is derived from the accesses below (as the reference does)
            ml = re.search(rf"const idx_t {n}_left_halo_{d} = (\d+);", text)
            mr = re.search(rf"const idx_t {n}_right_halo_{d} = (\d+);", text)
            v["halo"][d] = [int(ml.group(1)) if ml else 0, int(mr.group(1)) if mr else 0]
    vindex = {v["name"]: i for i, v in enumerate(ir["vars"])}
    # ---- stages / parts ---------------------------------------------------------------------------------
    stage_pos = [(m.start(), m.group(1)) for m in re.finditer(r"//////// Stencil stage '(\w+)' //////", text)]
    part_iter = list(re.finditer(r"////// Stencil (scratch )?part '(\w+)' ([^\n]*?)//////", text))
    if not part_iter:
        raise EmitError("no parts found")
    # scratch parts hang off the non-scratch parts that need them, in evaluation order
    # (StencilPartBase::get_reqd_parts, /root/reference/src/kernel/lib/stencil_calc.cpp:74-77)
    children: dict = {}
    for m in re.finditer(r"^\s*(\w+)\.add_scratch_child\(&(\w+)\);", text, re.M):
        children.setdefault(m.group(1), []).append(m.group(2))
    ir["scratch_parts"] = []
    for pm in part_iter:
        is_scratch_part, pname, cond = bool(pm.group(1)), pm.group(2), pm.group(3)
        has_step_cond = "w/o step condition" not in cond
        has_dom_cond = "w/o domain condition" not in cond
        stage = None
        if not is_scratch_part:
            stage = [s for pos, s in stage_pos if pos < pm.start()][-1]
        body_start = text.index("static void calc_scalar(", pm.end())
        body_end = text.index("} // calc_scalar.", body_start)
        body = text[body_start:body_end]
        head = text[pm.end():body_start]
        if bool(re.search(r"_is_scratch = true", head)) != is_scratch_part:
            raise EmitError(f"part '{pname}': inconsistent scratch markers")
        dom_cond = None
        if has_dom_cond:
            mm = re.search(r"is_in_valid_domain\(.*?\n(?:.*?\n)*?\s*return (.*);", head)
            if not mm:
                raise EmitError(f"part '{pname}': cannot find its sub-domain expression")
            dom_cond = parse_domain_cond(mm.group(1), dd)
        part = {"name": pname, "stage": stage, "cond": dom_cond, "scratch": is_scratch_part, "children": children.get(pname, []),
                "fp_ops": int(re.search(r"_scalar_fp_ops = (\d+);", head).group(1)),
                "reads": int(re.search(r"_scalar_points_read = (\d+);", head).group(1)),
                "writes": int(re.search(r"_scalar_points_written = (\d+);", head).group(1)),
                "accesses": [], "stmts": [], "outputs": []}
        ptr = {}   # expr_tempN (pointer) -> var name
        ptr_re = r"auto\* (expr_temp\d+) = (?:core_data->|thread_core_data\.)var_(\w+)_core_p\.get\(\);"
        for m in re.finditer(ptr_re, body):
            ptr[m.group(1)] = m.group(2)
        acc_index: dict = {}

        def access(var: str, idx_text: str):
            idxs = [s for s in re.split(r",\s*(?![^()]*\))", idx_text.strip()) if s.strip()] if idx_text.strip() else []
            v = ir["vars"][vindex[var]]
            if len(idxs) != len(v["dims"]):
                raise EmitError(f"index count mismatch for var '{var}'")
            toff = 0
            offs = {}
            misc = []
            for d, it in zip(v["dims"], idxs):
                dim, off = parse_index(it, v["dims"])
                if d != step_dim and d not in dd:      # misc dim: constant index
                    if dim is not None:
                        raise EmitError(f"var '{var}': misc dim '{d}' indexed by an expression ('{it}')")
                    misc.append(off)
                    rng = v.setdefault("misc_range", {}).setdefault(d, [off, off])
                    rng[0], rng[1] = min(rng[0], off), max(rng[1], off)
                    continue
                if dim is None:
                    raise EmitError(f"var '{var}': constant index '{it}' in non-misc dim '{d}'")
                if dim != d:
                    raise EmitError(f"var '{var}': index '{it}' does not follow declared dim '{d}'")
                if d == step_dim:
                    toff = off
                else:
                    offs[d] = off
            if len(misc) > 2:
                raise EmitError("more than 2 misc dims per var are not supported")
            key = (var, toff, tuple(misc))
            if key not in acc_index:
                acc_index[key] = len(part["accesses"])
                part["accesses"].append({"var": var, "toff": toff, "misc": misc})
            return acc_index[key], [offs.get(d, 0) for d in dd]

        READ_RE = r"(expr_temp\d+)->read_elem\(\{([^}]*)\}, \w+\)"

        def tmp_name(tok: str) -> str:
            """expr_temp12 -> e12, arg0_temp3 -> a0_3, res_temp14 -> r14 (names of the generated scalars)"""
            m = re.fullmatch(r"(expr|res|arg(\d+))_temp(\d+)", tok)
            return {"expr": "e", "res": "r"}.get(m.group(1), f"a{m.group(2)}_") + m.group(3)

        def parse_rhs(rhs_text: str):
            reads = []

            def repl(mm):
                a, offs = access(ptr[mm.group(1)], mm.group(2))
                reads.append((a, offs))
                return f"@{len(reads) - 1}"

            return Parser(re.sub(READ_RE, repl, rhs_text)).parse(), reads

        # step condition (IF_STEP): a boolean over the step index and, possibly, elements of (misc-dim) vars;
        # evaluated inside the kernel so that conditions on var contents need no host round trip
        if has_step_cond:
            mm = re.search(r"is_in_valid_step\(.*?\n((?:.*?\n)*?)\s*return (.*);", head)
            if not mm:
                raise EmitError(f"part '{pname}': cannot find its step-condition expression")
            sc_ptr = {m.group(1): m.group(2) for m in re.finditer(ptr_re, mm.group(1))}   # its own temp numbering
            sc_reads = []

            def sc_repl(m2):
                a, offs = access(sc_ptr[m2.group(1)], m2.group(2))
                sc_reads.append((a, offs))
                return f"@{len(sc_reads) - 1}"

            ctext = re.sub(READ_RE, sc_repl, mm.group(2))
            ctext = re.sub(rf"(?<![\w@]){step_dim}(?!\w)", "GT", ctext)
            left = re.sub(r"@\d+|GT|\d+(?:\.\d*)?(?:[eE][-+]?\d+)?|[-+*/%()<>=!&| ]", "", ctext)
            if left:
                raise EmitError(f"unsupported token(s) '{left}' in step condition of part '{pname}'")
            part["step_cond"] = {"expr": ctext, "reads": sc_reads,
                                 "text": re.search(r"w/step condition '(.*)'", cond).group(1)}

        for line in body.splitlines():
            line = line.strip()
            if not line or line.startswith("//"):
                continue
            m = re.fullmatch(r"real_t ((?:arg\d+|res|expr)_temp\d+) = (.*);", line)
            if m:
                if re.fullmatch(r"arg\d+_temp\d+", m.group(1)) and m.group(2).strip() == "0":
                    continue        # declaration of a multi-result function's output (set by the call below)
                tree, reads = parse_rhs(m.group(2))
                part["stmts"].append({"dst": tmp_name(m.group(1)), "tree": tree, "reads": reads})
                continue
            m = re.fullmatch(r"yask_(cos_and_sin|sin_and_cos)\((arg\d+_temp\d+), (arg\d+_temp\d+), (.*)\);", line)
            if m:
                tree, reads = parse_rhs(m.group(4))
                first, second = tmp_name(m.group(2)), tmp_name(m.group(3))
                cs = (first, second) if m.group(1) == "cos_and_sin" else (second, first)
                part["stmts"].append({"kind": "sincos", "cos": cs[0], "sin": cs[1], "tree": tree, "reads": reads})
                continue
            m = re.fullmatch(r"(expr_temp\d+)->write_elem\(((?:arg\d+|res|expr)_temp\d+), \{([^}]*)\}, \w+\);", line)
            if m:
                a, offs = access(ptr[m.group(1)], m.group(3))
                if any(offs):
                    raise EmitError("write with a spatial offset is not supported")
                part["outputs"].append({"access": a, "src": tmp_name(m.group(2))})
                continue
            if re.match(r"(static void calc_scalar|host_assert|auto& thread_core_data|idx_t \w+ = idxs|auto\* expr_temp|const auto step_temp)", line):
                continue
            raise EmitError(f"unrecognised statement in calc_scalar of {pname}: {line[:120]}")
        if not part["outputs"]:
            raise EmitError(f"part {pname} writes nothing")
        part["stmts"] = contract_like_gcc(part)
        if is_scratch_part:
            # write halo = largest halo of the scratch vars it writes (find_scratch_write_halos, setup.cpp:1182-1228)
            vmap = {v["name"]: v for v in ir["vars"]}
            wh = [[0, 0] for _ in dd]
            for o in part["outputs"]:
                ov = vmap[part["accesses"][o["access"]]["var"]]
                if not ov["scratch"]:
                    raise EmitError(f"scratch part '{pname}' writes the non-scratch var '{ov['name']}'")
                for i, d in enumerate(dd):
                    h = ov["halo"].get(d, [0, 0])
                    wh[i] = [max(wh[i][0], h[0]), max(wh[i][1], h[1])]
            part["wh"] = wh
            ir["scratch_parts"].append(part)
            continue
        st = next((s for s in ir["stages"] if s["name"] == stage), None)
        if st is None:
            st = {"name": stage, "parts": []}
            ir["stages"].append(st)
        st["parts"].append(part)
    return ir


# ----------------------------------------------------------------------------------------------------
# back-ends
# ----------------------------------------------------------------------------------------------------
def _const_text(tok: str) -> str:
    return tok if re.search(r"[.eE]", tok) else tok + ".0"


def gen_expr(tree, rd, ops) -> str:
    k = tree[0]
    if k == "const":
        return f"C({_const_text(tree[1])})"
    if k == "tmp":
        return tree[1]
    if k == "call":
        return f"YF_{tree[1]}(" + ", ".join(gen_expr(a, rd, ops) for a in tree[2]) + ")"
    if k == "read":
        return rd(tree[1])
    if k == "neg":
        return f"(-{gen_expr(tree[1], rd, ops)})"
    if k in ("mad", "msb", "nmad", "nmsb"):
        return f"{ops[k]}({gen_expr(tree[1], rd, ops)}, {gen_expr(tree[2], rd, ops)}, {gen_expr(tree[3], rd, ops)})"
    a, b = gen_expr(tree[1], rd, ops), gen_expr(tree[2], rd, ops)
    return f"{ops[k]}({a}, {b})"


# MAD(a,b,c) = a*b + c, MSB(a,b,c) = a*b - c, NMAD(a,b,c) = c - a*b, NMSB(a,b,c) = -(a*b) - c: the places where the reference's DEFAULT build fuses a
# multiplication into the addition that consumes it (contract_like_gcc below).  In fp_mode 0 they expand to the two
# separately rounded operations, otherwise to one fma -- nothing is left to nvcc's own contraction heuristics.
OPS = {'add': 'ADD', 'sub': 'SUB', 'mul': 'MUL', 'div': 'DIV', 'mad': 'MAD', 'msb': 'MSB', 'nmad': 'NMAD', 'nmsb': 'NMSB'}


def contract_like_gcc(part):
    """Rewrite the statement trees of `part` with the FMA contraction GCC applies to the reference's generated code in its
    default build (-O3, -ffp-contract=fast; tree-ssa-math-opts.c, convert_mult_to_fma): walking the operations in
    evaluation order, a multiplication is fused iff EVERY use of its value is an addition or subtraction that has not been
    turned into an FMA already; it is then fused into each of them and disappears.  (So of two products feeding one addition
    the one evaluated EARLIER is fused, the other stays a multiplication: for separate statements that is statement order, for
    a*b + c*d written inline it is c*d -- operands of the reference's overloaded operators are evaluated right to left.)  Values are numbered structurally first, as GCC's redundancy
    elimination does before that pass: the same product written twice is one value with two uses.
    Returns the new statement list; statements whose product was fused away are dropped."""
    nodes = {}          # value key -> node
    order = []          # nodes in evaluation order (first occurrence)

    class N:
        __slots__ = ("kind", "args", "leaf", "users", "dead", "name")

        def __init__(self, kind, args=(), leaf=None):
            self.kind, self.args, self.leaf, self.users, self.dead, self.name = kind, list(args), leaf, [], False, None

    named = {}          # temp name -> node

    def intern(kind, args, leaf=None):
        ids = [id(a) for a in args]
        key = (kind, tuple(sorted(ids)) if kind in ("add", "mul") else tuple(ids), leaf)
        n = nodes.get(key)
        if n is None:
            n = N(kind, args, leaf)
            nodes[key] = n
            order.append(n)
            for a in args:
                a.users.append(n)
        return n

    def build(tree, st):
        k = tree[0]
        if k == "const":
            return intern("const", (), ("c", float(tree[1])))
        if k == "tmp":
            if tree[1] not in named:
                raise EmitError(f"temp '{tree[1]}' used before its definition")
            return named[tree[1]]
        if k == "read":
            a, o = st["reads"][tree[1]]
            return intern("read", (), ("r", a, tuple(o)))
        if k == "call":
            return intern("call", [build(a, st) for a in tree[2]], ("f", tree[1]))
        if k == "neg":
            return intern("neg", [build(tree[1], st)])
        # operands of an operator written inline are evaluated RIGHT first (they are arguments of the reference's overloaded
        # real_vec_t operators, which GCC evaluates right to left); pinned by wave2d's default-build fixtures
        r_ = build(tree[2], st)
        l_ = build(tree[1], st)
        return intern(k, [l_, r_])

    roots = []
    uid = [0]
    for st in part["stmts"]:
        if st.get("kind") == "sincos":
            arg = build(st["tree"], st)
            uid[0] += 1
            sc = N("sincos", [arg], ("sc", uid[0]))     # two results, never merged with anything
            arg.users.append(sc)
            order.append(sc)
            for nm in (st["sin"], st["cos"]):
                leaf = N("scres", [sc], ("scres", nm))
                sc.users.append(leaf)
                named[nm] = leaf
            roots.append((st, sc))
            continue
        r = build(st["tree"], st)
        named[st["dst"]] = r
        if r.name is None:
            r.name = st["dst"]
        roots.append((st, r))
    sink = N("out")
    for o in part["outputs"]:
        named[o["src"]].users.append(sink)
    # step conditions read temps? (no: they read vars only)
    for n in order:
        if n.kind != "mul" or not n.users:
            continue
        # uses: additions / subtractions, possibly through a negation that has that single use
        # (convert_mult_to_fma: "a negate on the multiplication leads to FNMA")
        sites = []      # (value seen by the add/sub, the add/sub, negated?)
        ok = True
        for u in n.users:
            if u.kind == "neg" and len(u.users) == 1 and u.users[0].kind in ("add", "sub"):
                sites.append((u, u.users[0], True))
            elif u.kind in ("add", "sub"):
                sites.append((n, u, False))
            else:
                ok = False
        if not ok or any(t.args[0] is v and t.args[1] is v for v, t, _ in sites) or len({id(t) for _, t, _ in sites}) != len(sites):
            continue
        a, b = n.args
        for v, u, negd in sites:
            left = u.args[0] is v
            other = u.args[1] if left else u.args[0]
            if u.kind == "add":
                kind = "nmad" if negd else "mad"                      # other - a*b | a*b + other
            elif left:
                kind = "nmsb" if negd else "msb"                      # -(a*b) - other | a*b - other
            else:
                kind = "mad" if negd else "nmad"                      # other + a*b | other - a*b
            u.kind, u.args = kind, [a, b, other]
            a.users.append(u); b.users.append(u)
            if negd:
                v.dead = True
        n.dead = True
    # back to trees: a node that is the root of a (live) statement is referred to by that statement's name
    def tree_of(n, top):
        if not top and n.name is not None and not n.dead:
            return ("tmp", n.name)
        if n.kind == "const":
            return ("const", repr(n.leaf[1]))
        if n.kind == "read":
            return ("readx", n.leaf[1], n.leaf[2])
        if n.kind == "scres":
            return ("tmp", n.leaf[1])
        if n.kind == "call":
            return ("call", n.leaf[1], [tree_of(a, False) for a in n.args])
        if n.kind == "neg":
            return ("neg", tree_of(n.args[0], False))
        if n.kind in ("mad", "msb", "nmad", "nmsb"):
            return (n.kind, tree_of(n.args[0], False), tree_of(n.args[1], False), tree_of(n.args[2], False))
        return (n.kind, tree_of(n.args[0], False), tree_of(n.args[1], False))

    def with_reads(tree, reads):
        """("readx", acc, offs) leaves -> ("read", index into this statement's read list)"""
        k = tree[0]
        if k == "readx":
            reads.append((tree[1], list(tree[2])))
            return ("read", len(reads) - 1)
        if k in ("const", "tmp"):
            return tree
        if k == "call":
            return ("call", tree[1], [with_reads(a, reads) for a in tree[2]])
        return (k,) + tuple(with_reads(a, reads) for a in tree[1:])

    def finish(d, tree):
        reads = []
        d["tree"] = with_reads(tree, reads)
        d["reads"] = reads
        return d

    out = []
    emitted = set()
    for st, r in roots:
        if st.get("kind") == "sincos":
            out.append(finish({"kind": "sincos", "sin": st["sin"], "cos": st["cos"]}, tree_of(r.args[0], False)))
            continue
        if r.dead:
            continue                      # fused into its users
        if r.name != st["dst"]:
            out.append(finish({"dst": st["dst"]}, ("tmp", r.name) if r.name else tree_of(r, True)))     # alias of an earlier value
            continue
        if id(r) in emitted:
            continue
        emitted.add(id(r))
        out.append(finish({"dst": st["dst"]}, tree_of(r, True)))
    # outputs may name a statement that was an alias of a fused product: cannot happen (a product written out has a
    # non-add use, so it is never fused)
    return out


def _rd_text(a, offs, masks):
    offs = [0] * (3 - len(offs)) + list(offs)     # domain dims are right-aligned into the kernel's (x,y,z) slots
    return f"RD({a}, {masks[a]}, {offs[0]}, {offs[1]}, {offs[2]})"


def _stmt_lines(part, ndd, indent="    ", masks=None):
    out = []
    for s in part["stmts"]:
        def rd(i, s=s):
            return _rd_text(*s["reads"][i], masks)
        if s.get("kind") == "sincos":
            out.append(f"{indent}T {s['sin']}, {s['cos']};")
            out.append(f"{indent}YF_sincos({gen_expr(s['tree'], rd, OPS)}, {s['sin']}, {s['cos']});")
            continue
        out.append(f"{indent}const T {s['dst']} = {gen_expr(s['tree'], rd, OPS)};")
    for o in part["outputs"]:
        out.append(f"{indent}WR({o['access']}, {masks[o['access']]}, {o['src']});")
    return out


def _cond_text(part, masks):
    """C text of the part's combined sub-domain and step conditions (None if unconditional)."""
    terms = []
    if part.get("cond"):
        terms.append(f"({part['cond']['expr']})")
    sc = part.get("step_cond")
    if sc:
        terms.append("(" + re.sub(r"@(\d+)", lambda m: "(double)" + _rd_text(*sc["reads"][int(m.group(1))], masks), sc["expr"]) + ")")
    return " && ".join(terms) if terms else None


def _cond_comment(part):
    c = []
    if part.get("cond"):
        c.append("sub-domain: " + part["cond"]["text"])
    if part.get("step_cond"):
        c.append("step condition: " + part["step_cond"]["text"])
    return "; ".join(c)


def _all_parts(ir):
    """Every part in evaluation order: (stage name or None, part).  Scratch parts first (table order = index)."""
    return [(None, p) for p in ir.get("scratch_parts", [])] + [(st["name"], p) for st in ir["stages"] for p in st["parts"]]


def _stage_sequence(ir, st):
    """Evaluation order of one stage: each part preceded by the scratch parts it requires that have not been
    evaluated yet in this stage (parts_done, /root/reference/src/kernel/lib/stencil_calc.cpp:118-127)."""
    smap = {p["name"]: p for p in ir.get("scratch_parts", [])}
    svars = {v["name"] for v in ir["vars"] if v.get("scratch")}

    def reads_of(p):
        outs = {o["access"] for o in p["outputs"]}
        return {a["var"] for i, a in enumerate(p["accesses"]) if i not in outs and a["var"] in svars}

    def writes_of(p):
        return {p["accesses"][o["access"]]["var"] for o in p["outputs"]}

    seq, done = [], set()
    for p in st["parts"]:
        # The reference lists every scratch part a part depends on, directly or through OTHER NON-SCRATCH parts; only
        # those reachable through scratch vars are needed to evaluate it (the others were evaluated for the part that
        # reads them), so the rest is skipped here.
        needed, frontier = set(), reads_of(p)
        while frontier:
            needed |= frontier
            nxt = set()
            for c in p.get("children", []):
                if writes_of(smap[c]) & frontier:
                    nxt |= reads_of(smap[c]) - needed
            frontier = nxt
        for c in p.get("children", []):
            if not (writes_of(smap[c]) & needed):
                continue
            if c not in done:
                done.add(c)
                seq.append(smap[c])
        seq.append(p)
    return seq



# ----------------------------------------------------------------------------------------------------
# sweep kernels (TMA-staged shared-memory planes, warp-specialised; yask_b200/csrc/yb_gen_sweep.cuh)
# ----------------------------------------------------------------------------------------------------
SWEEP_SMEM_LIMIT = 225 * 1024          # of the 227 KB a CTA may use
SWEEP_TWO_CTA_SMEM = 112 * 1024        # two CTAs per SM below this
SWEEP_MAX_STREAMS = 28
SWEEP_XQUEUE = os.environ.get("YB_EMIT_SWEEP_XQ", "1") != "0"     # x neighbours of split streams in registers (tuning knob)


def _roundup(v, m):
    return (v + m - 1) // m * m


def _sweep_streams(ir, p, ty, pf):
    """TMA streams of part `p` for a tile of `ty` rows x 32 vectors and `pf` planes of prefetch, or None when the part does
    not qualify (3-D solutions, unconditional non-scratch parts, full-rank outputs, no misc-dim / scratch vars among the
    full-rank reads).  A var whose x neighbours are only read at the point's own (y, z) may be SPLIT into the current plane
    with its y/z halo ('H') and a ring of halo-less planes ('C'); chosen when that needs less shared memory."""
    if len(ir["domain_dims"]) != 3 or p.get("cond") or p.get("step_cond") or p.get("scratch") or p.get("children"):
        return None
    masks = _masks(ir, p)
    if any(masks[o["access"]] != 7 for o in p["outputs"]):
        return None
    vmap = {v["name"]: v for v in ir["vars"]}
    eb = ir["elem_bytes"]
    vw = 16 // eb
    tz = 32 * vw
    offs = {}
    for st in p["stmts"]:
        for a, o in st["reads"]:
            offs.setdefault(a, set()).add(tuple(o))
    streams = []

    def mk(a, kind, xl, xr, pts):
        yl = min(o[1] for o in pts); yr = max(o[1] for o in pts)
        zl = min(o[2] for o in pts); zr = max(o[2] for o in pts)
        # The box must START on a 16-byte boundary in global memory (pads and tile origins are multiples of 128 B, so only
        # the z reach matters): measured on B200 -- UTMALDG raises "illegal instruction" for a start coordinate that is not
        # a multiple of 16 B.  The vector loads of the consumers need the same alignment on both ends.
        zl = -_roundup(-zl, vw)
        zr = _roundup(zr, vw)
        rows = ty + yr - yl
        pz = tz + zr - zl
        slot = _roundup(rows * pz * eb, 128)
        ns = xr - xl + 1 + pf
        return {"acc": a, "kind": kind, "xl": xl, "xr": xr, "yl": yl, "yr": yr, "zl": zl, "zr": zr, "rows": rows, "pz": pz,
                "slot": slot, "ns": ns, "bytes": rows * pz * eb}

    for a in sorted(offs):
        if masks[a] != 7:
            continue
        acc = p["accesses"][a]
        if acc.get("misc") or vmap[acc["var"]].get("scratch"):
            return None
        pts = offs[a]
        xl, xr = min(o[0] for o in pts), max(o[0] for o in pts)
        whole = [mk(a, "W", xl, xr, pts)]
        star = all(o[1] == 0 and o[2] == 0 for o in pts if o[0] != 0)
        here = [o for o in pts if o[0] == 0]
        choice = whole
        if star and here and xr - xl + 1 >= 3 and any(o[1] or o[2] for o in here):
            split = [mk(a, "H", 0, 0, here), mk(a, "C", xl, xr, [(0, 0, 0)])]
            if sum(s_["ns"] * s_["slot"] for s_ in split) < sum(s_["ns"] * s_["slot"] for s_ in whole):
                choice = split
        streams += choice
    if not streams or len(streams) > SWEEP_MAX_STREAMS:
        return None
    off = 0
    for s_ in streams:
        s_["off"] = off
        off += s_["ns"] * s_["slot"]
    return streams, off


def sweep_plan(ir, p):
    """Tile shape, prefetch depth and shared-memory layout of part `p`'s sweep kernel, or None.  Always 8 consumer warps:
    a tile of 8 rows gives every thread one 16-byte vector of points, a tile of 4 rows (rings of 8 rows do not fit) half
    a vector -- two warps then share a tile row."""
    # (tile rows, consumer warps, planes of prefetch).  4-row tiles (one or two points per thread, two warps per scheduler) are
    # latency-bound and take a third plane of prefetch when it fits: ssg fp64 512^3 +5.8 % on one box (profiles/r2_generated.md).
    # A fourth plane (fits ssg's stage 1) measured no further gain.
    cands = [(8, 8, 2), (4, 8, 3), (4, 8, 2), (8, 8, 1), (4, 8, 1)]
    if os.environ.get("YB_EMIT_SWEEP_TY"):                          # tuning knobs: force one candidate
        ty = int(os.environ["YB_EMIT_SWEEP_TY"])
        cands = [(ty, int(os.environ.get("YB_EMIT_SWEEP_NW", "8")), int(os.environ.get("YB_EMIT_SWEEP_PF", "2")))]
    for ty, nw, pf in cands:
        r = _sweep_streams(ir, p, ty, pf)
        if r is None:
            return None
        streams, ring_bytes = r
        bar_off = _roundup(ring_bytes, 8)
        smem = bar_off + 16 * (pf + 1)
        if smem > SWEEP_SMEM_LIMIT:
            continue
        eb = ir["elem_bytes"]
        vw = 16 // eb
        tz = 32 * vw
        nwz = max(1, nw // ty)                     # warps per tile row
        tv = vw // nwz                             # points per thread (a 16-byte vector, or a part of one)
        if tv < 1 or ty * nwz != nw:
            continue
        # One CTA per SM (8 + 4 warps, up to 168 registers per thread at launch): launch with enough dynamic shared memory
        # that a second CTA never fits -- the consumers' setmaxnreg.inc below is sized for one resident CTA and would wait
        # forever for registers next to a second one.
        occ = 1
        smem_launch = max(smem, 117 * 1024)
        return {"ty": ty, "nw": nw, "nwz": nwz, "tv": tv, "rpt": 1, "pf": pf, "vw": vw, "tz": tz, "streams": streams, "bar_off": bar_off,
                "smem": smem, "smem_launch": smem_launch, "occ": occ, "threads": nw * 32 + 128,
                # consumer register budget after setmaxnreg (64 K registers per SM, producer warpgroup keeps 24 each)
                "cregs": min(232, ((65536 // occ - 128 * 24) // (nw * 32)) // 8 * 8),
                "bytes0": sum((s_["xr"] - s_["xl"] + 1) * s_["bytes"] for s_ in streams),
                "bytes1": sum(s_["bytes"] for s_ in streams)}
    return None


def emit_sweep_kernel(ir, p, plan, ident) -> list:
    masks = _masks(ir, p)
    T = "float" if ir["elem_bytes"] == 4 else "double"
    eb, vw, nw, rpt, pf = ir["elem_bytes"], plan["tv"], plan["nw"], plan["rpt"], plan["pf"]      # vw: points per THREAD from here on
    streams = plan["streams"]
    outs = {o["access"] for o in p["outputs"]}

    def stream_of(a, o):
        """Index of the stream that serves the read of access `a` at offset o = (dx, dy, dz)."""
        for k, s_ in enumerate(streams):
            if s_["acc"] != a:
                continue
            if s_["kind"] == "W" or (s_["kind"] == "H" and o[0] == 0) or (s_["kind"] == "C" and o[0] != 0):
                return k
        raise EmitError("read without a stream")

    # ---- classify the reads ---------------------------------------------------------------------------------
    loads = {}        # (k, dx, row offset, vector index) -> name
    hoist = {}        # (acc, (dx, dy, dz)) -> (where, name): lower-rank reads moved out of the point bodies
    for st in p["stmts"]:
        for a, o in st["reads"]:
            o = tuple(o)
            m = masks[a]
            if m == 7:
                k = stream_of(a, o)
                for i in range(vw):
                    j = (i + o[2]) // vw
                    loads.setdefault((k, o[0], o[1] - streams[k]["yl"], j), None)
            elif a not in outs and m in (0, 1, 2, 4):
                hoist.setdefault((a, o), None)
    # x neighbours in registers: a stream that is only read at the point's own (y, z) (long x reach) in a kernel whose threads own at most one 64-bit
    # value per plane is read ONCE per plane -- the newest -- into a per-thread queue that shifts by one plane per iteration
    # (the whole reach is read at the first iteration of a chunk, when the ring holds it).  The ring and the producer are
    # unchanged; this trades (reach - 1) shared-memory loads and their ring addresses for register moves.
    def own(k, ry, j):
        return ry == -streams[k]["yl"] and j == 0

    xq = {k for k, s_ in enumerate(streams)
          if s_["kind"] in "CW" and vw * eb <= 8 and rpt == 1 and s_["xr"] - s_["xl"] + 1 >= 4 and SWEEP_XQUEUE
          and all(own(k, ry, j) for (k2, dx, ry, j) in loads if k2 == k and dx != 0)}
    n_str = len({s_["acc"] for s_ in streams})
    # Points of a vector beyond the box are computed like the others (their reads stay inside shared memory / clamped
    # indices) and simply not stored -- unless the part has reads that go to global memory with the point's own indices.
    guard = any(masks[a] != 7 and (a, tuple(o)) not in hoist for st in p["stmts"] for a, o in st["reads"])
    L = []
    L.append(f"// sweep kernel of part '{p['name']}' (yb_gen_sweep.cuh): {len(streams)} TMA streams over {n_str} vars, tile {plan['ty']} rows x {plan['tz']} z, "
             f"{nw} consumer warps x {vw} point(s) per thread, {pf} planes of prefetch, {plan['smem']} B of shared memory, {plan['occ']} CTA(s) per SM")
    L.append("template <int MODE>")
    L.append(f"__global__ void __launch_bounds__({plan['threads']}, {plan['occ']}) {ident}_{p['name']}_sweep_kernel(const __grid_constant__ GenSweepParams SP) {{")
    L.append(f"    typedef {T} T;")
    L.append(f"    constexpr int VW = {vw}, NW = {nw}, NWZ = {plan['nwz']}, RPT = {rpt}, TY = {plan['ty']}, TZ = {plan['tz']}, PF = {pf}, NB = PF + 1;")
    L.append("    extern __shared__ __align__(128) unsigned char sw_smem[];")
    L.append("    const GenParams& P = SP.g;")
    L.append(f"    uint64_t* full_bar = reinterpret_cast<uint64_t*>(sw_smem + {plan['bar_off']});")
    L.append("    uint64_t* done_bar = full_bar + NB;")
    L.append("    const int sw_bz = int(blockIdx.x) % SP.nzb, sw_by = (int(blockIdx.x) / SP.nzb) % SP.nyb, sw_bc = int(blockIdx.x) / (SP.nzb * SP.nyb);")
    L.append("    const int z0 = P.zb + sw_bz * TZ, y0_ = P.yb + sw_by * TY, xs = P.xb + sw_bc * SP.lx;")
    L.append("    const int sw_len = min(SP.lx, P.xe - xs);")
    L.append("    if (threadIdx.x == 0) {")
    L.append("        for (int b = 0; b < NB; b++) { mbar_init(&full_bar[b], 1); mbar_init(&done_bar[b], NW); }")
    L.append("        fence_barrier_init();")
    L.append("    }")
    L.append("    __syncthreads();")
    L.append("    if (threadIdx.x >= NW * 32) {")
    L.append("        // ---- producer warpgroup: one lane streams every plane of this CTA, then exits ----")
    L.append('        asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");')
    L.append("        if (threadIdx.x == NW * 32) {")
    L.append("            int fb = 0, db = 0; unsigned dpar = 0;")
    L.append("            for (int j = 0; j < sw_len; j++) {")
    L.append("                if (j > PF) {       // the slots written now were last read at iteration j - 1 - PF")
    L.append("                    mbar_wait(&done_bar[db], dpar);")
    L.append("                    if (++db == NB) { db = 0; dpar ^= 1u; }")
    L.append("                }")
    L.append("                uint64_t* bar = &full_bar[fb];")
    L.append("                if (++fb == NB) fb = 0;")
    L.append(f"                mbar_arrive_expect_tx(bar, j == 0 ? {plan['bytes0']}u : {plan['bytes1']}u);")
    for k, s_ in enumerate(streams):
        acc = p["accesses"][s_["acc"]]
        L.append(f"                SW_ISSUE({k}, {s_['off']}, {s_['slot']}, {s_['ns']}, {s_['xl']}, {s_['xr']}, {s_['yl']}, {s_['zl']})   // {acc['var']}"
                 f"(t{acc['toff']:+d}) {s_['kind']}: x {s_['xl']}..{s_['xr']}, y {s_['yl']}..{s_['yr']}, z {s_['zl']}..{s_['zr']}")
    L.append("            }")
    L.append("        }")
    L.append("        return;")
    L.append("    }")
    L.append(f'    asm volatile("setmaxnreg.inc.sync.aligned.u32 {plan["cregs"]};");')
    L.append("    // ---- consumers: NWZ warps per tile row; a thread owns VW consecutive z points of its row ----")
    L.append("    const int lane = int(threadIdx.x) & 31, sw_w = int(threadIdx.x) >> 5, sw_r0 = (sw_w / NWZ) * RPT;")
    L.append("    const int zt = ((sw_w % NWZ) * 32 + lane) * VW;                   // z offset of this thread's points within the tile")
    L.append("    const int zq = z0 + zt;                                           // first z of this thread's points")
    L.append("    const int nzv = max(0, min(VW, P.ze - zq));                       // valid points of the vector")
    L.append("    const uint32_t sw_base = smem_u32(sw_smem);")
    for k, s_ in enumerate(streams):
        L.append(f"    const uint32_t t{k} = sw_base + {s_['off']}u + uint32_t((sw_r0 * {s_['pz']} + zt + {-s_['zl']}) * {eb});")
    # hoisted lower-rank reads that do not depend on x
    for (a, o) in sorted(hoist):
        m = masks[a]
        nm = f"h{a}_{'_'.join(('m' if c < 0 else 'p') + str(abs(c)) for c in o)}"
        if m == 0:
            hoist[(a, o)] = ("pre", nm)
            L.append(f"    const T {nm} = static_cast<const T*>(P.ptr[{a}])[0];")
        elif m == 2:
            hoist[(a, o)] = ("row", nm)
            L.append(f"    T {nm}[RPT];")
            L.append(f"    _Pragma(\"unroll\") for (int r = 0; r < RPT; r++) {nm}[r] = static_cast<const T*>(P.ptr[{a}])[(min(y0_ + sw_r0 + r, P.ye - 1) + ({o[1]})) * P.sy[{a}]];")
        elif m == 4:
            hoist[(a, o)] = ("vec", nm)
            L.append(f"    T {nm}[VW];")
            L.append(f"    _Pragma(\"unroll\") for (int i = 0; i < VW; i++) {nm}[i] = static_cast<const T*>(P.ptr[{a}])[(min(zq + i, P.ze - 1) + ({o[2]})) * P.sz[{a}]];")
        else:
            hoist[(a, o)] = ("plane", nm)
    # Ring positions: one byte offset per distinct (ring length, slot size) -- the offset of the slot that holds the OLDEST
    # plane of the ring (x + XL) -- advanced by one slot per iteration with a wrap; a plane `ahead` slots further is one add
    # and one conditional subtract away, shared by every stream with the same ring shape (no multiplications, no divisions).
    rings = sorted({(s_["ns"], s_["slot"]) for s_ in streams})
    L.append("    int fb = 0; unsigned fpar = 0;")
    L.append("    " + " ".join(f"uint32_t q{n}_{sl} = 0;" for n, sl in rings) + "      // byte offset of the oldest plane's slot, per ring shape")
    L.append("    const bool vec_ok = nzv == VW && ((reinterpret_cast<uintptr_t>(static_cast<T*>(P.ptr[%d]) + zq) & (VW * sizeof(T) - 1)) == 0) && (P.SY %% VW == 0) && (P.SX %% VW == 0);" % p["outputs"][0]["access"])
    for k in sorted(xq):
        s_ = streams[k]
        L.append("    " + " ".join(f"T xq{k}_{d}[VW] = {{}};" for d in range(s_["xr"] - s_["xl"] + 1)) + f"      // x queue of stream {k}: planes x{s_['xl']:+d} .. x{s_['xr']:+d}")
    L.append("    for (int it = 0; it < sw_len; it++) {")
    L.append("        mbar_wait(&full_bar[fb], fpar);")
    L.append("        const int x = xs + it;")
    for (a, o), (where, nm) in sorted(hoist.items()):
        if where == "plane":
            L.append(f"        const T {nm} = static_cast<const T*>(P.ptr[{a}])[(x + ({o[0]})) * P.sx[{a}]];")
    # plane bases per (stream, dx) actually read
    used = sorted({(k, dx) for (k, dx, ry, j) in loads if k not in xq or not own(k, ry, j)} | {(k, streams[k]["xr"]) for k in xq})
    rels = sorted({(streams[k]["ns"], streams[k]["slot"], dx - streams[k]["xl"]) for (k, dx) in used})
    for (n, sl, ahead) in rels:
        L.append(f"        const uint32_t r{n}_{sl}_{ahead} = " + (f"q{n}_{sl};" if ahead == 0 else f"sw_wrap(q{n}_{sl}, {ahead * sl}u, {n * sl}u);"))
    for (k, dx) in used:
        s_ = streams[k]
        L.append(f"        const uint32_t b{k}_{'m' if dx < 0 else 'p'}{abs(dx)} = t{k} + r{s_['ns']}_{s_['slot']}_{dx - s_['xl']};")
    for key in sorted(loads):
        k, dx, ry, j = key
        s_ = streams[k]
        nm = f"v{k}_{'m' if dx < 0 else 'p'}{abs(dx)}_{ry}_{'m' if j < 0 else 'p'}{abs(j)}"
        if k in xq and own(k, ry, j):
            nm = f"xq{k}_{dx - s_['xl']}"
        loads[key] = nm
    for k in sorted(xq):
        s_ = streams[k]
        nq = s_["xr"] - s_["xl"] + 1
        thr = f"uint32_t(({-s_['yl']} * {s_['pz']}) * {eb})"
        L.append("        if (it == 0) {")
        for d in range(nq):
            L.append(f"            SwVec<T, VW>::lds(t{k} + {d * s_['slot']}u + {thr}, xq{k}_{d});")
        L.append("        } else {")
        L.append("            _Pragma(\"unroll\") for (int i = 0; i < VW; i++) { " + " ".join(f"xq{k}_{d}[i] = xq{k}_{d + 1}[i];" for d in range(nq - 1)) + " }")
        L.append(f"            SwVec<T, VW>::lds(b{k}_{'m' if s_['xr'] < 0 else 'p'}{abs(s_['xr'])} + {thr}, xq{k}_{nq - 1});")
        L.append("        }")
    L.append("        _Pragma(\"unroll\") for (int r = 0; r < RPT; r++) {")
    L.append("            const int y = y0_ + sw_r0 + r;")
    for key in sorted(loads):
        k, dx, ry, j = key
        s_ = streams[k]
        if k in xq and own(k, ry, j):
            continue
        L.append(f"            T {loads[key]}[VW]; SwVec<T, VW>::lds(b{k}_{'m' if dx < 0 else 'p'}{abs(dx)} + uint32_t(((r + {ry}) * {s_['pz']} + ({j * vw})) * {eb}), {loads[key]});")
    for o in p["outputs"]:
        L.append(f"            T o{o['access']}[VW];")
    L.append("            if (y < P.ye) {")
    for i in range(vw):
        L.append((f"                if ({i} < nzv) {{" if guard else "                {") + f"        // point {i} of the vector")
        L.append(f"                    const int z = zq + {i}; (void)z;")

        def rd(ri, st=None, i=i):
            a, o = st["reads"][ri]
            o = tuple(o)
            if masks[a] == 7:
                k = stream_of(a, o)
                j = (i + o[2]) // vw
                c = (i + o[2]) % vw
                return f"{loads[(k, o[0], o[1] - streams[k]['yl'], j)]}[{c}]"
            if (a, o) in hoist:
                where, nm = hoist[(a, o)]
                return {"pre": nm, "plane": nm, "row": f"{nm}[r]", "vec": f"{nm}[{i}]"}[where]
            return _rd_text(a, o, masks)

        for st in p["stmts"]:
            rdf = (lambda ri, st=st: rd(ri, st))
            if st.get("kind") == "sincos":
                L.append(f"                    T {st['sin']}, {st['cos']};")
                L.append(f"                    YF_sincos({gen_expr(st['tree'], rdf, OPS)}, {st['sin']}, {st['cos']});")
                continue
            L.append(f"                    const T {st['dst']} = {gen_expr(st['tree'], rdf, OPS)};")
        for o in p["outputs"]:
            L.append(f"                    o{o['access']}[{i}] = {o['src']};")
        L.append("                }")
    for o in p["outputs"]:
        a = o["access"]
        L.append(f"                {{ T* dst = static_cast<T*>(P.ptr[{a}]) + (x * P.SX + y * P.SY + zq);")
        L.append(f"                  if (vec_ok) SwVec<T, VW>::stg(dst, o{a}); else for (int i = 0; i < nzv; i++) dst[i] = o{a}[i]; }}")
    L.append("            }")
    L.append("        }")
    L.append("        __syncwarp();")
    L.append("        if (lane == 0) mbar_arrive(&done_bar[fb]);      // this warp is done with the oldest slots")
    L.append("        if (++fb == NB) { fb = 0; fpar ^= 1u; }")
    L.append("        " + " ".join(f"q{n}_{sl} = sw_wrap(q{n}_{sl}, {sl}u, {n * sl}u);" for n, sl in rings))
    L.append("    }")
    L.append("}")
    return L


def _masks(ir, part):
    """Per access: bit k set if the var spans the domain dim held by kernel slot k (slots x=1, y=2, z=4; the
    solution's domain dims are right-aligned into the slots, so the unit-stride dim is always slot z)."""
    dd = ir["domain_dims"]
    sh = 3 - len(dd)
    vmap = {v["name"]: v for v in ir["vars"]}
    out = []
    for a in part["accesses"]:
        m = 0
        for i, d in enumerate(dd):
            if d in vmap[a["var"]]["dims"]:
                m |= 1 << (i + sh)
        # a var that declares its domain dims in another order than the solution (H(y, z, x)) is stored in ITS order:
        # bit 8 keeps it off the shared-geometry fast path (mask 7) -- it is addressed through its own strides
        vd = [d for d in vmap[a["var"]]["dims"] if d in dd]
        if vd != [d for d in dd if d in vd]:
            m |= 8
        out.append(m)
    return out


def emit_cuda(ir: dict) -> str:
    n = ir["name"]
    ident = c_ident(n)
    L = []
    L.append(f"// GENERATED by yask_b200/emitter/yask_cuda_emit.py from the reference compiler's analysis of solution '{n}'.")
    L.append("// Do not edit: re-run the emitter.  One kernel per solution part; statements are the part's expression")
    L.append("// tree in the reference's evaluation order (generated calc_scalar(), emitted by")
    L.append("// /root/reference/src/compiler/lib/YaskKernel.cpp:429- / Cpp.cpp), every op in the element type.")
    L.append("#pragma once")
    L.append('#include "../yb_gen_sweep.cuh"')
    L.append("namespace yb { namespace gen {")
    for stname, p in _all_parts(ir):
        where = f"of stage '{stname}'" if stname else "(scratch: evaluated over the box expanded by its write halo, before the parts that read it)"
        L.append(f"// part '{p['name']}' {where}: {p['fp_ops']} FP ops, {p['reads']} reads, {p['writes']} writes per point")
        L.append("template <typename T, int MODE>")
        L.append(f"__global__ void __launch_bounds__(GEN_BLOCK) {ident}_{p['name']}_kernel(const __grid_constant__ GenParams P) {{")
        L.append("    GEN_KERNEL_BEGIN")
        masks = _masks(ir, p)
        ct = _cond_text(p, masks)
        if ct:
            L.append(f"    if ({ct}) {{   // {_cond_comment(p)}")
        L.extend(_stmt_lines(p, len(ir["domain_dims"]), masks=masks))
        if ct:
            L.append("    }")
        L.append("    GEN_KERNEL_END")
        L.append("}")
    plans = {}
    for st in ir["stages"]:
        for p in st["parts"]:
            plan = sweep_plan(ir, p)
            if plan:
                plans[p["name"]] = plan
                L.extend(emit_sweep_kernel(ir, p, plan, ident))
    # spec table
    L.append(f"inline void {ident}_describe(GenStencil& g) {{")
    L.append(f'    g.name = "{n}"; g.elem_bytes = {ir["elem_bytes"]}; g.step_dim = "{ir["step_dim"]}";')
    L.append("    g.domain_dims = {" + ", ".join(f'"{d}"' for d in ir["domain_dims"]) + "};")
    for v in ir["vars"]:
        dims = ", ".join(f'"{d}"' for d in v["dims"])
        hl = ", ".join(str(v["halo"].get(d, [0, 0])[0]) for d in ir["domain_dims"])
        hr = ", ".join(str(v["halo"].get(d, [0, 0])[1]) for d in ir["domain_dims"])
        mr = v.get("misc_range", {})
        mf = ", ".join(str(mr[d][0]) if d in mr else "0" for d in v["dims"])
        ms = ", ".join(str(mr[d][1] - mr[d][0] + 1) if d in mr else "0" for d in v["dims"])
        L.append(f'    g.vars.push_back(GenVar{{"{v["name"]}", {{{dims}}}, {v["alloc_t"]}, {str(v["is_output"]).lower()}, {v["l1_norm"]}, {{{hl}}}, {{{hr}}}, {{{mf}}}, {{{ms}}}, {str(bool(v.get("scratch"))).lower()}}});')
    vidx = {v["name"]: i for i, v in enumerate(ir["vars"])}
    sh = 3 - len(ir["domain_dims"])
    for st in ir["stages"]:
        L.append(f'    g.stages.push_back(GenStage{{"{st["name"]}", {{}}}});')
        for p in _stage_sequence(ir, st):
            acc = ", ".join("{%d, %d, {%s}}" % (vidx[a["var"]], a["toff"], ", ".join(str(m) for m in (a.get("misc", []) + [0, 0])[:2])) for a in p["accesses"])
            outs = ", ".join(str(o["access"]) for o in p["outputs"])
            k = f"{ident}_{p['name']}_kernel"
            fns = f"{{{{GEN_FN({k}, float, 0), GEN_FN({k}, float, 1)}}, {{GEN_FN({k}, double, 0), GEN_FN({k}, double, 1)}}}}"
            bl = []
            bnds = (p.get("cond") or {}).get("bounds") or {}
            kind = {"0": 0, "GF": 1, "GL": 2}
            for d in range(3):
                lo, hi = bnds.get(str(d), [None, None])
                bl.append(f"{{{kind[lo[0]] if lo else -1}, {lo[1] if lo else 0}, {kind[hi[0]] if hi else -1}, {hi[1] if hi else 0}}}")
            wh = [[0, 0]] * sh + (p.get("wh") or [[0, 0]] * len(ir["domain_dims"]))     # right-aligned into the (x,y,z) slots
            whl = ", ".join(str(w[0]) for w in wh)
            whr = ", ".join(str(w[1]) for w in wh)
            conditional = str(bool(p.get("cond") or p.get("step_cond"))).lower()
            L.append(f'    g.stages.back().parts.push_back(GenPart{{"{p["name"]}", {p["fp_ops"]}, {p["reads"]}, {p["writes"]}, {{{acc}}}, {{{outs}}}, {fns}, {{{", ".join(bl)}}}, '
                     f'{str(p["scratch"]).lower()}, {conditional}, {{{whl}}}, {{{whr}}}}});')
            plan = plans.get(p["name"])
            if plan:
                ks = f"{ident}_{p['name']}_sweep_kernel"
                fi = 0 if ir["elem_bytes"] == 4 else 1
                L.append("    {")
                L.append("        GenSweep& sw = g.stages.back().parts.back().sweep;")
                L.append(f"        sw.fn[{fi}][0] = GEN_SW_FN({ks}, 0); sw.fn[{fi}][1] = GEN_SW_FN({ks}, 1);")
                L.append(f"        sw.ty = {plan['ty']}; sw.tz = {plan['tz']}; sw.threads = {plan['threads']}; sw.occ = {plan['occ']}; sw.smem = {plan['smem_launch']};")
                for s_ in plan["streams"]:
                    L.append("        sw.streams.push_back(GenSweepStream{%d, %d, %d, %d, %d, %d, %d, %d, %d, %d, %d, %d});" % (
                        s_["acc"], s_["xl"], s_["xr"], s_["yl"], s_["yr"], s_["zl"], s_["zr"], s_["rows"], s_["pz"], s_["slot"], s_["ns"], s_["off"]))
                L.append("    }")
    L.append("}")
    L.append("} }  // namespace yb::gen")
    return "\n".join(L) + "\n"


def emit_oracle(ir: dict) -> str:
    n = ir["name"]
    ident = c_ident(n)
    T = "float" if ir["elem_bytes"] == 4 else "double"
    L = []
    L.append(f"/* GENERATED by yask_b200/emitter/yask_cuda_emit.py -- TEST INFRASTRUCTURE ONLY (CPU oracle for '{n}').")
    L.append(" * Plain-C restatement of the statements the reference compiler emits for each part (generated")
    L.append(" * calc_scalar()), evaluated as the reference's VECTOR path does: constants rounded to the element")
    L.append(" * type, every operation in the element type, no contraction (compile with -ffp-contract=off).")
    L.append(" * Pinned against the reference built with -ffp-contract=off (tests/golden). */")
    for _, p in _all_parts(ir):
        L.append(f"static void yo_{ident}_{p['name']}(const yo_gen_args* A) {{")
        L.append(f"    typedef {T} T;")
        L.append("    YO_GEN_LOOP_BEGIN")
        masks = _masks(ir, p)
        ct = _cond_text(p, masks)
        if ct:
            L.append(f"        if ({ct}) {{   /* {_cond_comment(p)} */")
        L.extend(_stmt_lines(p, len(ir["domain_dims"]), indent="        ", masks=masks))
        if ct:
            L.append("        }")
        L.append("    YO_GEN_LOOP_END")
        L.append("}")
    L.append(f"static const yo_gen_part yo_{ident}_parts[] = {{")
    for _, p in _all_parts(ir):
        L.append(f'    {{"{p["name"]}", yo_{ident}_{p["name"]}, {len(p["accesses"])}}},')
    L.append("};")
    return "\n".join(L) + "\n"


def write_registry():
    """Regenerate the include lists / tables of every emitted solution from gen/manifest.json."""
    gdir = os.path.join(ROOT, "yask_b200", "csrc", "gen")
    odir = os.path.join(ROOT, "oracle", "gen")
    man = json.load(open(os.path.join(gdir, "manifest.json")))
    names = sorted(man)
    cu = ["// GENERATED by yask_b200/emitter/yask_cuda_emit.py: every emitted solution (see manifest.json).",
          "// Each solution is its own translation unit (gen/<name>.gen.cu) so that they compile in parallel."]
    cu += [f"namespace yb {{ namespace gen {{ void {c_ident(n)}_register(GenStencil& g); }} }}" for n in names]
    cu.append("#define YB_GEN_TABLE \\")
    cu += [f'    {{"{n}", yb::gen::{c_ident(n)}_register}}, \\' for n in names]
    cu.append("")
    open(os.path.join(gdir, "gen_all.inc"), "w").write("\n".join(cu) + "\n")
    for n in names:
        i = c_ident(n)
        open(os.path.join(gdir, f"{i}.gen.cu"), "w").write(
            f"// GENERATED: translation unit of solution '{n}'.\n#include \"{i}.gen.cuh\"\n"
            f"namespace yb {{ namespace gen {{ void {i}_register(GenStencil& g) {{ {i}_describe(g); }} }} }}\n")
    oc = ["/* GENERATED by yask_b200/emitter/yask_cuda_emit.py -- TEST INFRASTRUCTURE ONLY. */"]
    oc += [f'#include "{c_ident(n)}.gen.h"' for n in names]
    oc.append("#define YO_GEN_TABLE \\")
    oc += [f'    {{"{n}", yo_{c_ident(n)}_parts, (int)(sizeof(yo_{c_ident(n)}_parts) / sizeof(yo_gen_part))}}, \\' for n in names]
    oc.append("")
    open(os.path.join(odir, "gen_all.inc"), "w").write("\n".join(oc) + "\n")


def main(argv=None):
    if argv is None and "--all" in sys.argv[1:]:
        # re-emit every solution of the manifest (after an emitter change)
        man = json.load(open(os.path.join(ROOT, "yask_b200", "csrc", "gen", "manifest.json")))
        for name, m in sorted(man.items()):
            args = ["--stencil", m["stencil"], "--elem-bytes", str(m["elem_bytes"]), "--name", name, "--no-registry"]
            if m.get("radius"):
                args += ["--radius", str(m["radius"])]
            main(args)
        write_registry()
        return
    ap = argparse.ArgumentParser()
    ap.add_argument("--stencil", required=True)
    ap.add_argument("--elem-bytes", type=int, default=4)
    ap.add_argument("--radius", type=int, default=0)
    ap.add_argument("--name", default=None, help="registry name of the generated solution (default: stencil)")
    ap.add_argument("--no-registry", action="store_true", help="do not rewrite gen_all.inc (batch use)")
    ap.add_argument("--from-file", default=None, help="parse this already generated file instead of running the compiler")
    a = ap.parse_args(argv)
    name = a.name or a.stencil
    text = open(a.from_file).read() if a.from_file else run_frontend(a.stencil, a.elem_bytes, a.radius or None)
    ir = parse_generated(text, name)
    if ir["elem_bytes"] is None:
        ir["elem_bytes"] = a.elem_bytes
    ir["stencil"], ir["radius"] = a.stencil, a.radius
    gdir = os.path.join(ROOT, "yask_b200", "csrc", "gen")
    odir = os.path.join(ROOT, "oracle", "gen")
    os.makedirs(gdir, exist_ok=True)
    os.makedirs(odir, exist_ok=True)
    ident = c_ident(name)
    open(os.path.join(gdir, f"{ident}.gen.cuh"), "w").write(emit_cuda(ir))
    open(os.path.join(odir, f"{ident}.gen.h"), "w").write(emit_oracle(ir))
    slim = {k: v for k, v in ir.items() if k != "stages"}
    slim = {k: v for k, v in slim.items() if k != "scratch_parts"}
    table = [p["name"] for _, p in _all_parts(ir)]      # index of a part in the oracle's function table

    def slim_part(p):
        return {"name": p["name"], "index": table.index(p["name"]), "fp_ops": p["fp_ops"], "reads": p["reads"], "writes": p["writes"],
                "accesses": p["accesses"], "outputs": p["outputs"], "cond": p.get("cond"), "scratch": p["scratch"], "wh": p.get("wh"),
                "conditional": bool(p.get("cond") or p.get("step_cond")),
                "step_cond": (p.get("step_cond") or {}).get("text")}

    # "parts" of a stage = its evaluation sequence (required scratch parts first)
    slim["stages"] = [{"name": s["name"], "parts": [slim_part(p) for p in _stage_sequence(ir, s)]} for s in ir["stages"]]
    json.dump(slim, open(os.path.join(gdir, f"{name}.json"), "w"), indent=1)
    mpath = os.path.join(gdir, "manifest.json")
    man = json.load(open(mpath)) if os.path.exists(mpath) else {}
    man[name] = {"stencil": a.stencil, "radius": a.radius, "elem_bytes": ir["elem_bytes"]}
    json.dump(man, open(mpath, "w"), indent=1, sort_keys=True)
    if not a.no_registry:
        write_registry()
    nst = sum(len(p["stmts"]) for s in ir["stages"] for p in s["parts"])
    print(f"emitted {name}: {len(ir['vars'])} vars, {len(ir['stages'])} stage(s), {nst} statements, elem_bytes {ir['elem_bytes']}")


if __name__ == "__main__":
    main()
