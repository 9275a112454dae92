"""The AMGe V-cycle on the irregular hierarchies the benchmark spends its time on (tests/irregular_hierarchies.py): the
configs[4] deformed hexahedra (NullSpace dofs on level 1, rows of up to 179 entries, up to 55 colours), cube456
tetrahedra, and lognormal coefficients over four decades.  The uniform 8^3 hierarchy of the other V-cycle tests has
small, regular coarse levels and never reaches several SELL entry-group variants, colourings with 30-55 colours, or a
coarse PCG that really iterates.

P and D are the oracle's (fed through make_sequence), so every comparison tests the solve path, not Coarsen():
  a. the Galerkin level operators against the oracle's RAP;
  b. the colouring and standalone l1-GS / weighted GS sweeps on every level operator and every Hiptmair auxiliary
     operator, SELL (every group size, PDL on and off) and CSR, with the SELL variant counters against the host rules;
  c. the V-cycle in direct, graph and program mode against each other and the oracle (the mode is part of each id);
  d. the outer PCG of bench.py's solvers against the oracle's PCG."""
import numpy as np
import pytest

from oracle import drivers, solve as orc
from parelag_b200 import api, capi
from tests import irregular_hierarchies as IH
from tests.test_vcycle_modes_gpu import (SMOOTHERS, amge_entries, make_sequence, program_mode, rel, rhs_sequence, run_prec,
                                         tuning, with_sell)

pytestmark = pytest.mark.gpu

GS_SLOTS = {c: capi.sell_group_slot("gs", *c) for c in IH.CHOICES}
SPMV_SLOTS = {c: capi.sell_group_slot("spmv", *c) for c in IH.CHOICES}
CASES = [("deformed", 0), ("deformed", 1), ("deformed", 2), ("tets", 0), ("coefficients", 1), ("coefficients", 2)]


@pytest.fixture(scope="module")
def sess():
    return api.session()


@pytest.fixture(scope="module")
def hiers():
    """hierarchies built on first use and kept for the module"""
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = IH.build(name)
        return cache[name]
    return get


def counted(slots):
    c = capi.variant_counts()
    return {k: int(c[s]) for k, s in slots.items()}


# ------------------------------------------------------------------------------------------------------------------
# a: Galerkin levels
@pytest.mark.parametrize("name,form", CASES, ids=["%s-form%d" % c for c in CASES])
def test_galerkin_levels_match_oracle(sess, hiers, name, form):
    seqs, _, ess = hiers(name)
    ops = [A for lab, A in IH.level_operators(seqs, form, ess) if lab.endswith("-A")]
    S = make_sequence(seqs)
    solver = api.Solver(api.library_xml(drivers.library_entries(form)), "AMGe", ops[0], S, 0, form, ess)
    assert solver.num_levels() == len(seqs)
    for l in range(1, len(seqs)):
        Ag, Ao = solver.level_matrix(l), ops[l]
        assert np.array_equal(Ag.indptr, Ao.indptr), l
        assert np.array_equal(Ag.indices, Ao.indices), l
        assert np.max(np.abs(Ag.data - Ao.data)) <= 1e-12 * np.max(np.abs(Ao.data)), l
    solver.free(); S.free()


# ------------------------------------------------------------------------------------------------------------------
# b: colouring and standalone sweeps
SWEEPS = 2


def _sweep(sess, dA, stype, weights, b, x0, iterative=True):
    s = capi.Smoother(sess, dA, type=stype, sweeps=SWEEPS, damping=weights[0], omega=weights[1],
                      ordering=capi.GS_MULTICOLOR)
    dx, db = capi.Vec(sess, data=x0), capi.Vec(sess, data=b)
    capi.variant_counts(reset=True)
    s.apply(db, dx, iterative)
    out = dx.download(), counted(GS_SLOTS), s.order()
    s.free(); dx.free(); db.free()
    return out


def _max_rel(a, b):
    return np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)


def check_operator(sess, label, A):
    """colour order, l1-GS (SELL every group size and PDL on/off, CSR) and GS(0.9, 1.2) on one operator"""
    n = A.shape[0]
    rng = np.random.default_rng(n)
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    oorder, ncol = orc.multicolor_order(A)
    dA = capi.Mat.from_scipy(sess, A)
    ref = {2: orc.Smoother(A, type=2, sweeps=SWEEPS, order=oorder).apply(b, x0, True),
           6: orc.Smoother(A, type=6, sweeps=SWEEPS, damping=0.9, omega=1.2, order=oorder).apply(b, x0, True)}
    got = {}
    for kernel in ("sell", "csr"):
        for group in ((0, 4, 8, 12) if kernel == "sell" else (0,)):
            for pdl in (1, 0):
                with with_sell(kernel, SELL_GROUP=group, PDL=pdl):
                    for stype, w in ((2, (1.0, 1.0)), (6, (0.9, 1.2))):
                        x, cnt, (order, starts) = _sweep(sess, dA, stype, w, b, x0)
                        assert np.array_equal(order, oorder) and len(starts) == ncol + 1, (label, kernel)
                        # the SELL path runs l1-GS with unit weights; weighted GS always takes the CSR kernel
                        want = IH.gs_counts(A, forced=group) if (kernel == "sell" and stype == 2) else dict.fromkeys(IH.CHOICES, 0)
                        assert cnt == want, (label, kernel, group, stype, cnt, want)
                        got[(kernel, group, pdl, stype)] = x
    for stype in (2, 6):
        for kernel in ("sell", "csr"):
            base = got[(kernel, 0, 1, stype)]
            for k, x in got.items():
                if k[0] == kernel and k[3] == stype:
                    assert np.array_equal(x, base), (label, k)
            assert _max_rel(base, ref[stype]) <= 1e-13, (label, kernel, stype, _max_rel(base, ref[stype]))
    # weighted GS: one CSR kernel whatever the SELL setting
    assert np.array_equal(got[("sell", 0, 1, 6)], got[("csr", 0, 1, 6)]), label
    # zero initial guess on the SELL path: the first colour is computed inside the renumbering pass
    with with_sell("sell"):
        x, cnt, _ = _sweep(sess, dA, 2, (1.0, 1.0), b, x0, iterative=False)
    assert cnt == IH.gs_counts(A, zero_guess=True), label
    assert _max_rel(x, orc.Smoother(A, type=2, sweeps=SWEEPS, order=oorder).apply(b, x0, False)) <= 1e-13, label
    # SELL SpMV: the group variant of the natural-order copy, bit-identical across group sizes
    choice = IH.spmv_choice(A)
    ys = []
    for group in (0, 4, 8, 12):
        with tuning(SELL_GROUP=group):
            dx, dy = capi.Vec(sess, data=x0), capi.Vec(sess, n)
            capi.variant_counts(reset=True)
            dA.spmv(dx, dy, alpha=1.0, beta=0.0)
            cnt = counted(SPMV_SLOTS)
            ys.append(dy.download())
            dx.free(); dy.free()
        want = dict.fromkeys(IH.CHOICES, 0)
        if choice is not None:
            G, single, rows = IH.spmv_choice(A, group)
            want[(G, single)] = rows
        assert cnt == want, (label, group, cnt, want)
    assert all(np.array_equal(y, ys[0]) for y in ys)
    assert _max_rel(ys[0], orc.matvec(A, x0)) <= 1e-13, label
    dA.free()
    return choice


@pytest.mark.parametrize("name,form", CASES, ids=["%s-form%d" % c for c in CASES])
def test_colouring_and_sweeps_on_every_level_operator(sess, hiers, name, form):
    seqs, _, ess = hiers(name)
    for label, A in IH.level_operators(seqs, form, ess):
        check_operator(sess, "%s-form%d-%s" % (name, form, label), A)


def test_sweeps_on_a_narrow_operator(sess):
    """rows of 3 entries: the single-group G = 4 sweep, which no hierarchy operator reaches"""
    A = IH.tridiagonal()
    assert IH.gs_counts(A)[(4, True)] > 0
    check_operator(sess, "tridiagonal", A)


# ------------------------------------------------------------------------------------------------------------------
# c: execution modes
NCALLS = 4
SUBSET = [s for s in SMOOTHERS if (s[0], s[1], s[2]) in (("L1 Gauss-Seidel", "multicolor", "sell"),
                                                          ("L1 Gauss-Seidel", "multicolor", "csr"),
                                                          ("L1 Gauss-Seidel", "natural", "sell"),
                                                          ("L1 Jacobi", "natural", None))
          or (s[0] == "Chebyshev" and s[5] == 3)]
PRODUCTION = ("L1 Gauss-Seidel", "multicolor", "default-threshold", 1.0, 1.0, 2)


def _mode_cases():
    out = []
    for name, form in CASES:
        smoothers = SMOOTHERS if (name, form) == ("deformed", 2) else SUBSET
        for (sm, ordering, kernel, w, om, cheby) in list(smoothers) + [PRODUCTION]:
            if sm == "Lumped Jacobi" and form == 0:
                continue
            # As in test_vcycle_modes_gpu.py, Lumped Jacobi runs as a plain smoother.  So does Chebyshev on the deformed
            # hierarchy: its coarse auxiliary operators D^T A D have rows with a zero diagonal (the NullSpace dofs),
            # and Chebyshev scales by 1/sqrt(diag).
            hiptmair = form > 0 and sm != "Lumped Jacobi" and not (sm == "Chebyshev" and name == "deformed")
            # at the default threshold no level of these hierarchies (< 200 000 rows) takes the SELL kernel, so the
            # program has no op for the CSR sweep and falls back to the graph
            pm = "graph" if kernel == "default-threshold" else program_mode(sm, ordering, kernel)
            tag = "%s-%s-%s-w%g-om%g-cheb%d" % (sm.replace(" ", ""), ordering, kernel or "default", w, om, cheby)
            out.append(pytest.param(name, form, hiptmair, sm, ordering, kernel, w, om, cheby, pm,
                                    id="%s-form%d%s-%s-program_runs_as_%s" % (name, form, "-hiptmair" if hiptmair else "",
                                                                              tag, pm)))
    return out


@pytest.mark.parametrize("name,form,hiptmair,smoother,ordering,kernel,damping,omega,cheby,prog_mode", _mode_cases())
def test_execution_modes_match_direct_and_oracle(sess, hiers, name, form, hiptmair, smoother, ordering, kernel, damping,
                                                 omega, cheby, prog_mode):
    seqs, _, ess = hiers(name)
    A, marker = drivers.system_matrix(seqs[0], form, ess)
    rs = rhs_sequence(A.shape[0], marker, NCALLS, seed=200 + form)
    S = make_sequence(seqs)
    outs, modes = {}, {}
    with with_sell(None if kernel == "default-threshold" else kernel):
        for mode in ("direct", "graph", "program"):
            xml = api.library_xml(amge_entries(form, smoother, ordering, damping, omega, cheby, mode, hiptmair=hiptmair))
            solver = api.Solver(xml, "PCG-AMGe", A, S, 0, form, ess)
            outs[mode], modes[mode] = run_prec(sess, solver, rs)
            solver.free()
    S.free()
    assert modes["direct"] == ["direct"] * NCALLS
    assert modes["graph"] == ["direct"] + ["graph"] * (NCALLS - 1)
    assert modes["program"] == ["direct"] + [prog_mode] * (NCALLS - 1)
    H = drivers.amge_pcg_solver(seqs, form, ess, A, ordering=ordering, smoother_type=smoother, damping=damping,
                                omega=omega, cheby_order=cheby, hiptmair=hiptmair)
    tol = 1e-9 if smoother == "Chebyshev" else 1e-11
    for i, r in enumerate(rs):
        zo = H.mult(r)
        for mode in outs:
            assert rel(outs[mode][i], zo) <= tol, (mode, i, rel(outs[mode][i], zo))
        assert np.array_equal(outs["graph"][i], outs["direct"][i]), (i, rel(outs["graph"][i], outs["direct"][i]))
        if prog_mode == "graph":
            assert np.array_equal(outs["program"][i], outs["direct"][i]), i
        # The program's dot products use another reduction tree (PE_OP_DOT).  Here the coarse PCG really iterates, and
        # its coarse operators (NullSpace dofs, coefficients over four decades) amplify those last-bit differences:
        # measured on a B200 up to 1.1e-12 relative, against <= 1e-13 on the uniform 8^3 hierarchy.
        assert np.linalg.norm(outs["program"][i] - outs["direct"][i]) <= 1e-11 * np.linalg.norm(zo), \
            (i, rel(outs["program"][i], outs["direct"][i]))


# ------------------------------------------------------------------------------------------------------------------
# d: the benchmark's solvers
@pytest.mark.parametrize("kernel", ["default-threshold", "sell"])
@pytest.mark.parametrize("name,form", [("deformed", 2), ("deformed", 1), ("tets", 0)],
                         ids=["deformed-form2", "deformed-form1", "tets-form0"])
def test_bench_solver_pcg_matches_oracle(sess, hiers, name, form, kernel):
    import bench
    seqs, _, ess = hiers(name)
    A, marker = drivers.system_matrix(seqs[0], form, ess)
    b = np.random.default_rng(31 + form).standard_normal(A.shape[0])
    b[marker] = 0.0
    H = drivers.amge_pcg_solver(seqs, form, ess, A, ordering="multicolor")
    xo, ito, convo, histo = orc.pcg(A, H.mult, b, rtol=1e-6, atol=1e-6, max_iter=300)
    lib = bench.library_h1("multicolor") if form == 0 else bench.library("multicolor", form)
    S = make_sequence(seqs)
    with with_sell(None if kernel == "default-threshold" else kernel):
        solver = api.Solver(api.library_xml(lib), "PCG with Auxiliary Space Preconditioner", A, S, 0, form, ess)
        x = solver.mult(b)
        hist, it, conv = solver.history()
        solver.free()
    S.free()
    assert conv and convo and abs(it - ito) <= 1, (it, ito)
    m = min(len(hist), len(histo))
    ho = np.array(histo[:m])
    assert np.max(np.abs(hist[:m] - ho) / np.abs(ho)) < 1e-9
    assert np.linalg.norm(x - xo) <= 1e-8 * np.linalg.norm(xo)
