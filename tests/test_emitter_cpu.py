"""The CUDA emitter (yask_b200/emitter/yask_cuda_emit.py) re-run on the reference compiler's output must reproduce the
committed generated sources (kernels + oracle restatement) -- needs the reference's compiler, which oracle/build_ref.sh stages
under oracle/_ref/ship/refc;
plus parser unit checks that need no reference."""
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "yask_b200", "emitter"))
import yask_cuda_emit as E  # noqa: E402

GEN = os.path.join(ROOT, "yask_b200", "csrc", "gen")
MAN = json.load(open(os.path.join(GEN, "manifest.json")))


@pytest.mark.parametrize("name", ["awp_elastic", "ssg", "test_scratch_2d", "test_scratch_boundary_1d", "test_step_cond_1d", "test_func_1d",
                                  "test_reverse_2d", "iso3dfd_sponge", "wave2d"])
def test_emitter_reproduces_committed_sources(name):
    if not os.path.exists(E.COMPILER):
        pytest.skip("reference compiler not built (oracle/build_ref.sh)")
    m = MAN[name]
    text = E.run_frontend(m["stencil"], m["elem_bytes"], m.get("radius") or None)
    ir = E.parse_generated(text, name)
    ident = E.c_ident(name)
    assert E.emit_cuda(ir) == open(os.path.join(GEN, f"{ident}.gen.cuh")).read()
    assert E.emit_oracle(ir) == open(os.path.join(ROOT, "oracle", "gen", f"{ident}.gen.h")).read()


def test_manifest_matches_registry_and_json():
    inc = open(os.path.join(GEN, "gen_all.inc")).read()
    for name in MAN:
        assert f'{{"{name}", yb::gen::{E.c_ident(name)}_register}}' in inc
        ir = json.load(open(os.path.join(GEN, f"{name}.json")))
        idx = sorted(p["index"] for st in ir["stages"] for p in st["parts"])
        assert len(set(idx)) >= 1 and all(p["name"] for st in ir["stages"] for p in st["parts"])
        # scratch parts precede the part that needs them; scratch vars come last in the var table
        flags = [bool(v.get("scratch")) for v in ir["vars"]]
        assert flags == sorted(flags)
        for st in ir["stages"]:
            assert not st["parts"][-1]["scratch"]


def test_expression_parser_keeps_evaluation_order():
    t = E.Parser("expr_temp3 + @0 * 2.5 - (expr_temp4 / @1)").parse()
    assert t == ("sub", ("add", ("tmp", "e3"), ("mul", ("read", 0), ("const", "2.5"))), ("div", ("tmp", "e4"), ("read", 1)))
    t = E.Parser("yask_max(arg0_temp3, -1.5e+00) * yask_cbrt(@0)").parse()
    assert t == ("mul", ("call", "max", [("tmp", "a0_3"), ("const", "-1.5e+00")]), ("call", "cbrt", [("read", 0)]))
    with pytest.raises(E.EmitError):
        E.Parser("yask_tanh(@0)").parse()


def test_domain_condition_bounds():
    c = E.parse_domain_cond("((x >= (FIRST_INDEX(x) + 5)) && (x <= (LAST_INDEX(x) - 3)))", ["x"])
    assert c["bounds"] == {"2": [["GF", 5], ["GL", -3]]} and "G(2)" in c["expr"]
    c = E.parse_domain_cond("((x < (FIRST_INDEX(x) + 20)) || (y > 3))", ["x", "y"])
    assert c["bounds"] is None


def _part(stmts, outs):
    """A synthetic part: statements as (dst, expression text over reads @0.. @9); read k = access k at offset 0."""
    ps = []
    for dst, text in stmts:
        tree = E.Parser(text).parse()
        ps.append({"dst": dst, "tree": tree, "reads": [(k, [0, 0, 0]) for k in range(10)]})
    return {"stmts": ps, "outputs": [{"access": 20, "src": o} for o in outs]}


def _text(part):
    rd = lambda st: (lambda i: f"r{st['reads'][i][0]}")
    return {st["dst"]: E.gen_expr(st["tree"], rd(st), E.OPS) for st in E.contract_like_gcc(part)}


def test_contraction_follows_the_gcc_rule():
    """contract_like_gcc: the FMA formation of GCC's convert_mult_to_fma restated on the statement lists -- the oracle built
    from these lists matches the reference's DEFAULT build bit for bit (tests/test_oracle_golden.py), here the rule itself."""
    # of two products feeding one addition the one evaluated earlier is fused, the other stays a multiplication:
    # inline operands are evaluated right to left ...
    assert _text(_part([("e1", "@0 * @1 + @2 * @3")], ["e1"])) == {"e1": "MAD(r2, r3, MUL(r0, r1))"}
    # ... separate statements in statement order
    t = _text(_part([("e1", "@0 * @1"), ("e2", "@2 * @3"), ("e3", "expr_temp1 + expr_temp2")], ["e3"]))
    assert t == {"e2": "MUL(r2, r3)", "e3": "MAD(r0, r1, e2)"}
    # a product consumed by another product is not fused; the outer product is
    assert _text(_part([("e1", "@0 * @1 * @2 + @3")], ["e1"])) == {"e1": "MAD(MUL(r0, r1), r2, r3)"}
    # subtraction on either side, negation with a single use
    assert _text(_part([("e1", "@0 * @1 - @2")], ["e1"])) == {"e1": "MSB(r0, r1, r2)"}
    assert _text(_part([("e1", "@2 - @0 * @1")], ["e1"])) == {"e1": "NMAD(r0, r1, r2)"}
    assert _text(_part([("e1", "-(@0 * @1) + @2")], ["e1"])) == {"e1": "NMAD(r0, r1, r2)"}
    # a named product with two additive uses is fused into both and disappears; with a non-additive use it is kept everywhere
    t = _text(_part([("e1", "@0 * @1"), ("e2", "expr_temp1 + @2"), ("e3", "@3 - expr_temp1")], ["e2", "e3"]))
    assert t == {"e2": "MAD(r0, r1, r2)", "e3": "NMAD(r0, r1, r3)"}
    t = _text(_part([("e1", "@0 * @1"), ("e2", "expr_temp1 + @2"), ("e3", "expr_temp1 * @3")], ["e2", "e3"]))
    assert t == {"e1": "MUL(r0, r1)", "e2": "ADD(e1, r2)", "e3": "MUL(e1, r3)"}
    # the same product written twice is ONE value (redundancy elimination runs before FMA formation)
    t = _text(_part([("e1", "@0 * @1 + @2"), ("e2", "(@1 * @0) * @3")], ["e1", "e2"]))
    assert t["e1"] == "ADD(MUL(r0, r1), r2)" and t["e2"] == "MUL(MUL(r0, r1), r3)"
    # a product that is written out is never fused away
    t = _text(_part([("e1", "@0 * @1"), ("e2", "expr_temp1 + @2")], ["e1", "e2"]))
    assert t == {"e1": "MUL(r0, r1)", "e2": "ADD(e1, r2)"}
