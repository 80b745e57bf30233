"""GPU parity tests for iso3dfd through the C ABI (yask_b200.capi), bit-exact:
  * against the committed golden outputs of the unmodified reference (both its default GCC build and
    its -ffp-contract=off build),
  * against the CPU oracle on seeded inputs at sizes it finishes in seconds (ragged/odd sizes, all radii
    for the direct kernel, every FP mode, every tile shape of the TMA kernel),
  * TMA kernel vs direct kernel on the device at sizes the oracle cannot reach (checksum equality).
"""
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.helpers import GOLDEN, contract_mode_of, golden_cases, load_golden, regen_inputs
from yask_b200 import capi
from yask_b200.synth import hash_field, var_salt

pytestmark = pytest.mark.gpu


def run_gpu(n, steps, ins, radius=8, fp_mode=2, opts=None, ret_soln=False):
    s = capi.Solution("iso3dfd", radius=radius)
    s.set_overall_domain_size_vec(n)
    s.set_option("fp_mode", fp_mode)
    for k, v in (opts or {}).items():
        s.set_option(k, v)
    s.prepare_solution(0)
    p, v = s.get_var("p"), s.get_var("v")
    for t in (0, 1):
        f, l = p.halo_box(t)
        p.set_elements_in_slice(ins[("p", t)], f, l)
    f, l = v.halo_box(0)
    v.set_elements_in_slice(ins[("v", 0)], f, l)
    if steps:
        s.run_solution(0, steps - 1)
    tl = p.get_last_valid_step_index()
    f, l = p.domain_box(tl)
    out = p.get_elements_in_slice(f, l)
    if ret_soln:
        return out, s
    s.close()
    return out


def synth_inputs(n, seed, radius=8):
    h = radius
    return {("p", 0): hash_field(seed, var_salt("p", 0), (-h, -h, -h), [i + 2 * h for i in n], -1, 1),
            ("p", 1): hash_field(seed, var_salt("p", 1), (-h, -h, -h), [i + 2 * h for i in n], -1, 1),
            ("v", 0): hash_field(seed, var_salt("v", 0), (0, 0, 0), n, 0.05, 0.3)}


@pytest.mark.parametrize("kernel", ["tma", "direct"])
@pytest.mark.parametrize("path", golden_cases("iso3dfd_avx512") + golden_cases("iso3dfd-strict"))
def test_bit_exact_vs_reference_golden(path, kernel):
    meta, arrays = load_golden(path)
    ins = regen_inputs(meta)
    got = run_gpu(meta["n"], meta["steps"], ins, fp_mode=contract_mode_of(meta["ref_tag"]), opts={"kernel": kernel})
    ref = arrays[f"p.t{meta['vars']['p']['steps'][1]}"]
    assert got.shape == ref.shape
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


@pytest.mark.parametrize("fp_mode", [0, 1, 2])
@pytest.mark.parametrize("tile", [0, 1, 2, 3, 4, 5, 6, 7])
@pytest.mark.parametrize("n,steps,lx", [((40, 70, 150), 2, 16), ((17, 33, 65), 3, 7), ((64, 64, 128), 1, 128), ((9, 8, 16), 2, 4)])
def test_tma_kernel_vs_oracle(n, steps, lx, tile, fp_mode):
    ins = synth_inputs(n, 99)
    got = run_gpu(n, steps, ins, fp_mode=fp_mode, opts={"kernel": "tma", "tile": tile, "lx": lx})
    ref = O.iso3dfd_run(ins[("p", 0)], ins[("p", 1)], ins[("v", 0)], 8, steps, fp_mode)[8:-8, 8:-8, 8:-8]
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


@pytest.mark.parametrize("radius", [1, 2, 3, 4, 5, 6, 7, 8])
def test_direct_kernel_all_radii_vs_oracle(radius):
    n = (20, 18, 37)
    ins = synth_inputs(n, 5, radius)
    got = run_gpu(n, 2, ins, radius=radius, fp_mode=2, opts={"kernel": "direct"})
    h = radius
    ref = O.iso3dfd_run(ins[("p", 0)], ins[("p", 1)], ins[("v", 0)], radius, 2, 2)[h:-h, h:-h, h:-h]
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


@pytest.mark.parametrize("fp_mode", [0, 2])
@pytest.mark.parametrize("radius", [1, 2, 3, 4, 5, 6, 7])
def test_tma_kernel_other_radii_vs_oracle(radius, fp_mode):
    """The tiled kernel is instantiated for every radius 1..8 (default variant); same expression order as the oracle."""
    n = (37, 45, 150)
    ins = synth_inputs(n, 21, radius)
    got = run_gpu(n, 3, ins, radius=radius, fp_mode=fp_mode, opts={"kernel": "tma", "lx": 13})
    h = radius
    ref = O.iso3dfd_run(ins[("p", 0)], ins[("p", 1)], ins[("v", 0)], radius, 3, fp_mode)[h:-h, h:-h, h:-h]
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_empty_run_and_halo_untouched():
    n = (16, 16, 32)
    ins = synth_inputs(n, 3)
    out, s = run_gpu(n, 2, ins, ret_soln=True)
    p = s.get_var("p")
    # halo cells are never written by run_solution (context.cpp:251-256): they still hold the input
    tl = p.get_last_valid_step_index()
    f, l = p.halo_box(tl)
    full = p.get_elements_in_slice(f, l)
    src = ins[("p", tl % 2)]   # slot parity: API step tl lives in slot tl%2, initialised from API step tl%2
    mask = np.ones(full.shape, bool)
    mask[8:-8, 8:-8, 8:-8] = False
    assert np.array_equal(full[mask], src[mask])
    assert np.array_equal(full[8:-8, 8:-8, 8:-8], out)
    st = s.get_stats()
    assert st.num_steps_done == 2 and st.num_elements == 16 * 16 * 32 and st.kernel_launches == 2
    assert st.est_fp_ops_done == 2 * 61 * st.num_elements and st.elapsed_secs > 0
    s.close()


def test_device_hash_fill_matches_numpy_generator():
    n = (12, 10, 20)
    s = capi.Solution("iso3dfd")
    s.set_overall_domain_size_vec(n)
    s.prepare_solution(0)
    p, v = s.get_var("p"), s.get_var("v")
    p.fill_hash(1, 42, var_salt("p", 1), -1.0, 1.0)
    v.fill_hash(0, 42, var_salt("v", 0), 0.05, 0.3)
    f, l = p.halo_box(1)
    assert np.array_equal(p.get_elements_in_slice(f, l), hash_field(42, var_salt("p", 1), (-8, -8, -8), [i + 16 for i in n], -1, 1))
    f, l = v.halo_box(0)
    assert np.array_equal(v.get_elements_in_slice(f, l), hash_field(42, var_salt("v", 0), (0, 0, 0), n, 0.05, 0.3))
    s.close()


def test_auto_tuner_picks_a_variant_and_results_stay_exact():
    """run_auto_tuner_now: times the compiled sweep variants (data not preserved), keeps the fastest, clears the stats;
    a run with fresh data afterwards is still bit-exact vs the oracle."""
    n, steps, seed = (64, 48, 160), 2, 21
    s = capi.Solution("iso3dfd")
    s.set_overall_domain_size_vec(n)
    s.prepare_solution(0)
    rep = s.run_auto_tuner_now()
    assert "best: tile=" in rep and rep.count("ms/step") >= 6, rep
    assert s.get_stats().num_steps_done == 0
    assert int(s.get_option("tile")) in (0, 1, 4, 5, 6, 7)
    ins = {("p", t): hash_field(seed, var_salt("p", t), (-8, -8, -8), [i + 16 for i in n], -1, 1) for t in (0, 1)}
    vv = hash_field(seed, var_salt("v", 0), (0, 0, 0), n, 0.05, 0.3)
    p, v = s.get_var("p"), s.get_var("v")
    for t in (0, 1):
        p.set_elements_in_slice(ins[("p", t)], *p.halo_box(t))
    v.set_elements_in_slice(vv, *v.halo_box(0))
    s.run_solution(0, steps - 1)
    tl = p.get_last_valid_step_index()
    got = p.get_elements_in_slice(*p.domain_box(tl))
    ref = O.iso3dfd_run(ins[("p", 0)], ins[("p", 1)], vv, 8, steps, 2)[8:-8, 8:-8, 8:-8]
    s.close()
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    g = capi.Solution("awp_elastic", elem_bytes=0)
    g.set_overall_domain_size_vec((48, 40, 96))
    g.prepare_solution(0)
    rep = g.run_auto_tuner_now()
    assert "best: gen_pf=" in rep, rep
    g.close()


def test_device_reductions_match_numpy():
    """yk_var::reduce_elements_in_slice on the device (double accumulation, fixed order): sum / sum of squares to
    1e-12 relative, max / min exact, product on a small box; repeatable bit for bit."""
    n = (40, 36, 100)
    s = capi.Solution("iso3dfd")
    s.set_overall_domain_size_vec(n)
    s.prepare_solution(0)
    p = s.get_var("p")
    p.fill_hash(0, 5, var_salt("p", 0), -1.0, 1.0)
    p.fill_hash(1, 5, var_salt("p", 1), 0.5, 1.5)
    for first, last in (((0, 0, 0, 0), (0, 39, 35, 99)), ((0, -8, -8, -8), (1, 47, 43, 107)), ((1, 3, 5, 7), (1, 20, 9, 64)),
                        ((1, 10, 10, 10), (1, 10, 10, 10))):
        ref = np.concatenate([p.get_elements_in_slice((t,) + tuple(first[1:]), (t,) + tuple(last[1:])).astype(np.float64).ravel()
                              for t in range(first[0], last[0] + 1)])
        r = p.reduce_elements_in_slice(first, last)
        assert r["num"] == ref.size
        assert abs(r["sum"] - ref.sum()) <= 1e-12 * np.abs(ref).sum()
        assert abs(r["sum_squares"] - (ref * ref).sum()) <= 1e-12 * (ref * ref).sum()
        assert r["max"] == ref.max() and r["min"] == ref.min()
        assert r == p.reduce_elements_in_slice(first, last)
    small = ((1, 4, 4, 4), (1, 6, 6, 9))
    ref = p.get_elements_in_slice(*small).astype(np.float64).ravel()
    assert abs(p.reduce_elements_in_slice(*small)["product"] - np.prod(ref)) <= 1e-12 * abs(np.prod(ref))
    s.close()


@pytest.mark.parametrize("n,steps", [((256, 256, 256), 3), ((300, 130, 200), 2), ((1024, 1024, 1024), 2)])   # last: BASELINE.json's full size
def test_tma_equals_direct_on_device_large(n, steps):
    """Size-independent property: both kernels evaluate the same expression tree, so their results
    must be bit-identical at any size; compared by an order-independent checksum plus a sub-box vs
    the CPU oracle."""
    sums = []
    sub = None
    for kern in ("tma", "direct"):
        s = capi.Solution("iso3dfd")
        s.set_overall_domain_size_vec(n)
        s.set_option("kernel", kern)
        s.prepare_solution(0)
        p, v = s.get_var("p"), s.get_var("v")
        for t in (0, 1):
            p.fill_hash(t, 7, var_salt("p", t), -1.0, 1.0)
        v.fill_hash(0, 7, var_salt("v", 0), 0.05, 0.3)
        s.run_solution(0, steps - 1)
        tl = p.get_last_valid_step_index()
        sums.append(p.checksum(tl))
        if kern == "tma":
            sub = p.get_elements_in_slice([tl, 100, 60, 90], [tl, 131, 91, 153])
        s.close()
    assert sums[0] == sums[1]
    # sub-box check against the oracle: recompute a haloed neighbourhood (steps*8 wider) from the generator
    m = 8 * steps
    lo = (100 - m, 60 - m, 90 - m)
    shp = (32 + 2 * m, 32 + 2 * m, 64 + 2 * m)
    ins0 = hash_field(7, var_salt("p", 0), [a - 8 for a in lo], [a + 16 for a in shp], -1, 1)
    ins1 = hash_field(7, var_salt("p", 1), [a - 8 for a in lo], [a + 16 for a in shp], -1, 1)
    vv = hash_field(7, var_salt("v", 0), lo, shp, 0.05, 0.3)
    ref = O.iso3dfd_run(ins0, ins1, vv, 8, steps, 2)[8:-8, 8:-8, 8:-8]
    assert np.array_equal(sub.view(np.uint32), ref[m:-m, m:-m, m:-m].view(np.uint32))


@pytest.mark.parametrize("tag,fp_mode", [("iso3dfd.avx512", 2), ("iso3dfd-strict.avx512", 0)])
@pytest.mark.parametrize("steps", [1, 2, 10])
def test_config1_live_reference_128(tag, fp_mode, steps):
    """BASELINE.json config 1 as written: iso3dfd order 16 fp32 128^3, one rank, against the UNMODIFIED reference on
    identical inputs, bit for bit (the default build against fp_mode 2, the -ffp-contract=off build against fp_mode 0).
    The reference's outputs are stored as the SHA-256 of their bytes and a seeded sample of points
    (tests/golden/iso3dfd_config1_128.json, written by `tests/golden/make_golden.py config1`)."""
    ref = json.load(open(os.path.join(GOLDEN, "iso3dfd_config1_128.json")))[f"{tag}/{steps}"]
    n = (128, 128, 128)
    ins = synth_inputs(n, 1234)
    for kernel in ("tma", "direct"):
        got = run_gpu(n, steps, ins, fp_mode=fp_mode, opts={"kernel": kernel})
        assert list(got.shape) == ref["shape"]
        assert got.view(np.uint32).ravel()[ref["index"]].tolist() == ref["bits"], kernel
        assert hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest() == ref["sha256"], kernel


def test_fuse_vars_shares_storage_between_solutions():
    """yk_var::fuse_vars / yk_solution::fuse_vars (aux/yk_var_api.hpp:1370-1397): after fusing, both vars address ONE device
    allocation -- a second solution steps the first one's data in place; incompatible layouts are refused."""
    n, seed = (40, 24, 64), 5
    ins = synth_inputs(n, seed)
    ref = O.iso3dfd_run(ins[("p", 0)], ins[("p", 1)], ins[("v", 0)], 8, 2, 2)[8:-8, 8:-8, 8:-8]
    _, a = run_gpu(n, 0, ins, ret_soln=True)          # holds the inputs, never runs
    b = capi.Solution("iso3dfd")
    b.set_overall_domain_size_vec(n)
    b.prepare_solution(0)
    for name in ("p", "v"):
        b.get_var(name).fuse_vars(a.get_var(name))
    assert b.get_var("p").device_ptr(0) == a.get_var("p").device_ptr(0)
    b.run_solution(0, 1)
    b.sync()
    pa = a.get_var("p")
    # `a` never ran: read its storage through b's step window (the data is shared, the bookkeeping is per solution)
    pb = b.get_var("p")
    tl = pb.get_last_valid_step_index()
    got = pb.get_elements_in_slice(*pb.domain_box(tl))
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    raw_a = pa.get_elements_in_slice(*pa.domain_box(tl % 2))     # same slot of the shared allocation
    assert np.array_equal(raw_a.view(np.uint32), ref.view(np.uint32))
    c = capi.Solution("iso3dfd")
    c.set_overall_domain_size_vec((n[0] + 8, n[1], n[2]))
    c.prepare_solution(0)
    with pytest.raises(capi.YaskError):
        c.get_var("p").fuse_vars(a.get_var("p"))
    b.close()                                         # the allocation lives on while `a` references it
    assert np.array_equal(pa.get_elements_in_slice(*pa.domain_box(tl % 2)).view(np.uint32), ref.view(np.uint32))
    a.close()
    c.close()


def test_var_checks_of_the_reference_var_test():
    """What the reference's src/kernel/tests/var_test.cpp checks, through the public API (that file itself includes the
    reference's internal headers and cannot be built against any public API): two scalar vars hold the same value after
    set_element; two padded 3-D vars exchange a sequence of values element by element and by slice
    (host buffer), over the whole allocation including the pads, and read back identically."""
    import ctypes as C
    L = capi.lib()
    s = capi.Solution("iso3dfd")
    s.set_rank_domain_size_vec((3, 5, 7))                    # var_test.cpp: 3 + 2*i points per dim
    a0, a1 = s.new_var("var1", []), s.new_var("var2", [])
    a3, b3 = s.new_var("var3", ["x", "y", "z"]), s.new_var("var4", ["x", "y", "z"])
    for d in range(3):                                       # min pad 1, 2, 3 as in var_test.cpp (the engine rounds z up to a 128-B line)
        for v in (a3, b3):
            capi._chk(L.yb_var_set_min_pad(s._h, v.index, d, 1 + d, 1 + d))
    s.prepare_solution(0)
    # 0-D
    for v in (a0, a1):
        v.set_elements_in_slice(np.array([3.14], np.float32), [], [])
    assert a0.get_elements_in_slice([], []).ravel()[0] == a1.get_elements_in_slice([], []).ravel()[0] == np.float32(3.14)
    # 3-D: a sequence of values over the first var's whole allocation
    ia, ib = a3.info, b3.info
    first = [ia.dims[k].rank_offset - ia.dims[k].left_pad for k in range(3)]
    last = [ia.dims[k].rank_offset + ia.dims[k].domain_size + ia.dims[k].right_pad - 1 for k in range(3)]
    shape = [l - f + 1 for f, l in zip(first, last)]
    seq = (1.0 + np.arange(int(np.prod(shape)), dtype=np.float32)).reshape(shape)
    a3.set_elements_in_slice(seq, first, last)
    # the box both vars hold: the second var's allocation is at least its pads 1,2,3 around the domain
    f2 = [max(first[k], ib.dims[k].rank_offset - ib.dims[k].left_pad) for k in range(3)]
    l2 = [min(last[k], ib.dims[k].rank_offset + ib.dims[k].domain_size + ib.dims[k].right_pad - 1) for k in range(3)]
    assert all(f2[k] <= -1 - k and l2[k] >= ib.dims[k].domain_size + k for k in range(3))
    # by slice
    b3.set_all_elements_same(-1.0)
    buf = a3.get_elements_in_slice(f2, l2)
    b3.set_elements_in_slice(buf, f2, l2)
    assert np.array_equal(b3.get_elements_in_slice(f2, l2), seq[tuple(slice(f2[k] - first[k], l2[k] - first[k] + 1) for k in range(3))])
    # element by element (a diagonal of points incl. pad cells)
    b3.set_all_elements_same(-1.0)
    for i in range(-1, 3):
        pt = [i, i, i]
        val = a3.get_elements_in_slice(pt, pt)
        b3.set_elements_in_slice(val, pt, pt)
        assert b3.get_elements_in_slice(pt, pt).ravel()[0] == seq[tuple(pt[k] - first[k] for k in range(3))]
    s.close()


def test_in_run_auto_tuner_keeps_results_exact():
    """yk_solution::reset_auto_tuner(true) / -auto_tune: while enabled every run_solution() step runs with the next launch
    variant and is timed; the steps are REAL steps (all variants compute the same bits), so a run that tunes on the way is
    still bit-exact vs the oracle; afterwards the tuner is off and a variant is selected."""
    n, seed = (64, 48, 160), 3
    ins = synth_inputs(n, seed)
    _, s = run_gpu(n, 0, ins, ret_soln=True)
    s.reset_auto_tuner(True)
    assert s.is_auto_tuner_enabled()
    steps = 18 * 3 + 4          # 18 variants x (1 cold + 2 timed) samples, then a few steps with the winner
    s.run_solution(0, steps - 1)
    assert not s.is_auto_tuner_enabled()
    rep = s.auto_tuner_report()
    assert rep.count("ms/step") == 18 and "<- best" in rep, rep
    p = s.get_var("p")
    tl = p.get_last_valid_step_index()
    got = p.get_elements_in_slice(*p.domain_box(tl))
    s.close()
    ref = O.iso3dfd_run(ins[("p", 0)], ins[("p", 1)], ins[("v", 0)], 8, steps, 2)[8:-8, 8:-8, 8:-8]
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
