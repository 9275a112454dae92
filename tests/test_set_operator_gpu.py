"""SetOperator on a built AMGe solver (api.Solver.set_operator, pe_api_solver_set_operator): new values on the same
sparsity pattern, as a time step of M + dt K brings them.  The update must leave the solver in the state a fresh
BuildSolver on the new operator produces with the same sequence, parameters and boundary labels: the Galerkin products
of the numeric-only pass are bit-identical to the two-pass product's, so every level matrix and every V-cycle output is
compared bit for bit with a solver built directly on the new operator, and with the oracle to the tolerances of
test_vcycle_modes_gpu.py.  A refused update (new pattern or size, a changed FixZeroRows row set, a blocked operator)
changes nothing."""
import numpy as np
import pytest

from oracle import drivers, solve as orc
from parelag_b200 import api, capi
from tests.test_vcycle_modes_gpu import (SMOOTHERS, amge_entries, make_sequence, program_mode, rel, rhs_sequence, run_prec,
                                         with_sell)

pytestmark = pytest.mark.gpu

ESS = np.ones(6, dtype=np.int32)


@pytest.fixture(scope="module")
def sess():
    return api.session()


@pytest.fixture(scope="module")
def hier():
    from oracle import amge
    return amge.build_hierarchy((8, 8, 8), 3)[1]


def scaled(A, marker, seed):
    """S A S on A's pattern: S a seeded positive diagonal, 1 on the essential rows"""
    s = np.random.default_rng(seed).uniform(0.5, 2.0, A.shape[0])
    s[marker] = 1.0
    B = A.tocsr().copy()
    rows = np.repeat(np.arange(B.shape[0]), np.diff(B.indptr))
    B.data = B.data * s[rows] * s[B.indices]
    return B


def levels(solver):
    return [solver.level_matrix(l) for l in range(solver.num_levels())]


def assert_same_levels(got, want):
    assert len(got) == len(want)
    for l, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g.indptr, w.indptr) and np.array_equal(g.indices, w.indices), l
        assert np.array_equal(g.data, w.data), (l, np.abs(g.data - w.data).max())


def _cases():
    out = []
    for form in (0, 1, 2):
        for (name, ordering, kernel, w, om, cheby) in SMOOTHERS:
            hiptmair = form > 0 and name != "Lumped Jacobi"
            if name == "Lumped Jacobi" and form == 0:
                continue
            tag = "%s-%s-%s-w%g-om%g-cheb%d" % (name.replace(" ", ""), ordering, kernel or "default", w, om, cheby)
            out.append(pytest.param(form, hiptmair, name, ordering, kernel, w, om, cheby,
                                    id="form%d%s-%s" % (form, "-hiptmair" if hiptmair else "", tag)))
    return out


NBEFORE, NAFTER = 3, 6


# ------------------------------------------------------------------------------------------------------------------
# 1 + 2: an update reaches the state of a fresh build, in direct and graph mode, and (multicolour SELL) as the program
@pytest.mark.parametrize("form,hiptmair,smoother,ordering,kernel,damping,omega,cheby", _cases())
def test_update_matches_fresh_build(sess, hier, form, hiptmair, smoother, ordering, kernel, damping, omega, cheby):
    seqs = hier
    A1, marker = drivers.system_matrix(seqs[0], form, ESS)
    A2 = scaled(A1, marker, seed=40 + form)
    rs = rhs_sequence(A1.shape[0], marker, NBEFORE + NAFTER, seed=200 + form)
    S = make_sequence(seqs)
    pm = program_mode(smoother, ordering, kernel)
    outs, modes, lev = {}, {}, {}
    with with_sell(kernel):
        for mode in ("direct", "graph", "program"):
            xml = api.library_xml(amge_entries(form, smoother, ordering, damping, omega, cheby, mode, hiptmair=hiptmair))
            upd = api.Solver(xml, "PCG-AMGe", A1, S, 0, form, ESS)
            before, _ = run_prec(sess, upd, rs[:NBEFORE])
            upd.set_operator(capi.Mat.from_scipy(sess, A2))
            outs[mode, "upd"], modes[mode, "upd"] = run_prec(sess, upd, rs[NBEFORE:])
            lev[mode, "upd"] = levels(upd)
            upd.free()
            fresh = api.Solver(xml, "PCG-AMGe", capi.Mat.from_scipy(sess, A2), S, 0, form, ESS)
            outs[mode, "fresh"], modes[mode, "fresh"] = run_prec(sess, fresh, rs[NBEFORE:])
            lev[mode, "fresh"] = levels(fresh)
            fresh.free()
            assert not any(np.array_equal(b, a) for b, a in zip(before, outs[mode, "upd"]))
    S.free()
    # the recorded cycle was dropped: direct, then recorded again
    assert modes["direct", "upd"] == ["direct"] * NAFTER
    assert modes["graph", "upd"] == ["direct"] + ["graph"] * (NAFTER - 1)
    assert modes["program", "upd"] == ["direct"] + [pm] * (NAFTER - 1)
    for mode in ("direct", "graph", "program"):
        assert modes[mode, "upd"] == modes[mode, "fresh"]
        assert_same_levels(lev[mode, "upd"], lev[mode, "fresh"])
    H = drivers.amge_pcg_solver(seqs, form, ESS, A2, ordering=ordering, smoother_type=smoother, damping=damping,
                                omega=omega, cheby_order=cheby, hiptmair=hiptmair)
    tol = 1e-9 if smoother == "Chebyshev" else 1e-11
    for i, r in enumerate(rs[NBEFORE:]):
        zo = H.mult(r)
        for mode in ("direct", "graph"):
            assert np.array_equal(outs[mode, "upd"][i], outs[mode, "fresh"][i]), (mode, i)
        assert np.array_equal(outs["graph", "upd"][i], outs["direct", "upd"][i]), i
        assert np.linalg.norm(outs["program", "upd"][i] - outs["direct", "upd"][i]) <= 1e-13 * np.linalg.norm(zo), i
        for mode in ("direct", "graph", "program"):
            assert rel(outs[mode, "upd"][i], zo) <= tol, (mode, i, rel(outs[mode, "upd"][i], zo))
    # consecutive outputs differ: no replay returned a stale result
    assert all(not np.array_equal(outs["graph", "upd"][i], outs["graph", "upd"][i + 1]) for i in range(NAFTER - 1))


# ------------------------------------------------------------------------------------------------------------------
# pre- and post-smoother as two Hiptmair objects (two factories): each computes and keeps its own auxiliary operator
def test_distinct_pre_and_post_hiptmair(sess, hier):
    seqs = hier
    form = 2
    A1, marker = drivers.system_matrix(seqs[0], form, ESS)
    A2 = scaled(A1, marker, seed=31)
    rs = rhs_sequence(A1.shape[0], marker, 4, seed=32)
    S = make_sequence(seqs)
    e = amge_entries(form, "L1 Gauss-Seidel", "multicolor", 1.0, 1.0, 2, "graph")
    e["Hiptmair-post"] = e["Hiptmair-GS-GS"]
    e["AMGe"][1]["PostSmoother"] = "Hiptmair-post"
    xml = api.library_xml(e)
    res = {}
    with with_sell("sell"):
        upd = api.Solver(xml, "PCG-AMGe", A1, S, 0, form, ESS)
        run_prec(sess, upd, rs)
        upd.set_operator(capi.Mat.from_scipy(sess, A2))
        res["upd"] = run_prec(sess, upd, rs) + (levels(upd),)
        upd.free()
        fresh = api.Solver(xml, "PCG-AMGe", A2, S, 0, form, ESS)
        res["fresh"] = run_prec(sess, fresh, rs) + (levels(fresh),)
        fresh.free()
    S.free()
    assert res["upd"][1] == res["fresh"][1] == ["direct"] + ["graph"] * 3
    for o, f in zip(res["upd"][0], res["fresh"][0]):
        assert np.array_equal(o, f)
    assert_same_levels(res["upd"][2], res["fresh"][2])


# ------------------------------------------------------------------------------------------------------------------
# 3: PCG after an update: history, iterations and convergence of a fresh build, and of the oracle PCG on A2;
# the other operator of the same mesh (other coefficients) as well as S A S
def other_coefficients(seq, form, marker, A1, seed):
    """alpha M_form + beta D^T M_{form+1} D on A1's pattern (the sum is formed entry by entry on A1's pattern)"""
    rng = np.random.default_rng(seed)
    a, b = rng.uniform(0.5, 2.0, 2)
    M = seq.mass_operator(form) if form > 0 else None
    D = seq.D[form]
    K = (D.T @ seq.mass_operator(form + 1) @ D).tocsr()
    B = A1.tocsr().copy()
    rows = np.repeat(np.arange(B.shape[0]), np.diff(B.indptr))
    vals = b * np.asarray(K[rows, B.indices]).ravel()
    if M is not None:
        vals = vals + a * np.asarray(M.tocsr()[rows, B.indices]).ravel()
    ess = marker[rows] | marker[B.indices]
    vals[ess] = 0.0
    vals[ess & (rows == B.indices)] = 1.0
    B.data = vals
    return B


@pytest.mark.parametrize("form,which", [(0, "scaled"), (1, "scaled"), (2, "scaled"), (2, "coefficients")])
def test_pcg_after_update(sess, hier, form, which):
    seqs = hier
    A1, marker = drivers.system_matrix(seqs[0], form, ESS)
    A2 = scaled(A1, marker, seed=7) if which == "scaled" else other_coefficients(seqs[0], form, marker, A1, seed=8)
    rng = np.random.default_rng(9)
    b = rng.standard_normal(A1.shape[0])
    b[marker] = 0.0
    S = make_sequence(seqs)
    xml = api.library_xml(amge_entries(form, "L1 Gauss-Seidel", "multicolor", 1.0, 1.0, 2, "graph"))
    with with_sell("sell"):
        upd = api.Solver(xml, "PCG-AMGe", A1, S, 0, form, ESS)
        upd.mult(b)
        upd.set_operator(capi.Mat.from_scipy(sess, A2))
        x_upd = upd.mult(b)
        h_upd = upd.history()
        upd.free()
        fresh = api.Solver(xml, "PCG-AMGe", A2, S, 0, form, ESS)
        x_fresh = fresh.mult(b)
        h_fresh = fresh.history()
        fresh.free()
    S.free()
    assert np.array_equal(x_upd, x_fresh)
    assert np.array_equal(h_upd[0], h_fresh[0]) and h_upd[1:] == h_fresh[1:]
    H = drivers.amge_pcg_solver(seqs, form, ESS, A2, ordering="multicolor")
    xo, ito, convo, histo = orc.pcg(A2, H.mult, b, rtol=1e-6, atol=1e-6, max_iter=300)
    assert (h_upd[1], h_upd[2]) == (ito, convo)
    assert np.all(np.abs(h_upd[0] - np.array(histo)) <= 1e-9 * np.abs(np.array(histo)))
    assert rel(x_upd, xo) <= 1e-9


# ------------------------------------------------------------------------------------------------------------------
# 4: A1 -> A2 -> A1 reproduces the solver built on A1
def test_round_trip(sess, hier):
    seqs = hier
    form = 1
    A1, marker = drivers.system_matrix(seqs[0], form, ESS)
    A2 = scaled(A1, marker, seed=11)
    rs = rhs_sequence(A1.shape[0], marker, 4, seed=12)
    S = make_sequence(seqs)
    xml = api.library_xml(amge_entries(form, "L1 Gauss-Seidel", "multicolor", 1.0, 1.0, 2, "graph"))
    with with_sell("sell"):
        s = api.Solver(xml, "PCG-AMGe", A1, S, 0, form, ESS)
        ref, _ = run_prec(sess, s, rs)
        lev_ref = levels(s)
        s.set_operator(capi.Mat.from_scipy(sess, A2))
        mid, _ = run_prec(sess, s, rs)
        s.set_operator(capi.Mat.from_scipy(sess, A1))
        back, modes = run_prec(sess, s, rs)
        lev_back = levels(s)
        s.free()
    S.free()
    assert modes == ["direct"] + ["graph"] * 3
    assert not np.array_equal(mid[0], ref[0])
    for o, r in zip(back, ref):
        assert np.array_equal(o, r)
    assert_same_levels(lev_back, lev_ref)


# ------------------------------------------------------------------------------------------------------------------
# 5: refusals name their reason and leave the solver computing what it computed
def zero_coarse_row(seqs, form, marker, A1):
    """S = 0 on the fine rows of the support of one column of the level-1 P (one without essential rows): that coarse
    row of P^T A P becomes zero"""
    P = seqs[0].get_P(form, ESS).tocsc()
    for c in range(P.shape[1]):
        rows = P.indices[P.indptr[c]:P.indptr[c + 1]][P.data[P.indptr[c]:P.indptr[c + 1]] != 0]
        if len(rows) and not marker[rows].any():
            break
    s = np.ones(A1.shape[0])
    s[rows] = 0.0
    B = A1.tocsr().copy()
    r = np.repeat(np.arange(B.shape[0]), np.diff(B.indptr))
    B.data = B.data * s[r] * s[B.indices]
    return B


def test_refusals_change_nothing(sess, hier):
    import scipy.sparse as sp
    seqs = hier
    form = 2
    A1, marker = drivers.system_matrix(seqs[0], form, ESS)
    rs = rhs_sequence(A1.shape[0], marker, 3, seed=21)
    S = make_sequence(seqs)
    xml = api.library_xml(amge_entries(form, "L1 Gauss-Seidel", "multicolor", 1.0, 1.0, 2, "graph"))
    i = int(np.flatnonzero(~marker)[0])
    stored = set(A1.indices[A1.indptr[i]:A1.indptr[i + 1]])
    j = next(k for k in np.flatnonzero(~marker) if k not in stored)
    coo = A1.tocoo()
    extra = sp.csr_matrix((np.append(coo.data, 1e-3), (np.append(coo.row, i), np.append(coo.col, j))), shape=A1.shape)
    n = A1.shape[0]
    bigger = sp.block_diag([A1, sp.identity(1)]).tocsr()
    cases = [("extra entry", extra, "sparsity pattern"), ("size", bigger, "size"),
             ("zero rows", zero_coarse_row(seqs, form, marker, A1), "zero rows")]
    with with_sell("sell"):
        s = api.Solver(xml, "PCG-AMGe", A1, S, 0, form, ESS)
        ref, _ = run_prec(sess, s, rs)
        for what, B, reason in cases:
            with pytest.raises(capi.PEError, match=reason):
                s.set_operator(capi.Mat.from_scipy(sess, B))
            again, _ = run_prec(sess, s, rs)
            for o, r in zip(again, ref):
                assert np.array_equal(o, r), what
        s.free()
    S.free()
    assert n == A1.shape[0]


def test_block_solver_refuses(sess, hier):
    S = api.Sequence.hex((8, 8, 8), 3, jstart=2)
    M, B, Bt = S.assemble_darcy(sess, 0)
    nu, npr = M.info()[0], B.info()[0]
    b = np.random.default_rng(5).standard_normal(nu + npr)
    Mh = M.to_scipy()
    xml = api.library_xml(drivers.darcy_library_entries(block="Block GS", amge=True))
    solver = api.BlockSolver(xml, "GMRES-AMGe-Blk", [[M, Bt], [B, None]], S, 0, [2, 3])
    x = solver.mult(b)
    with pytest.raises(capi.PEError, match="MfemBlockOperator"):
        solver.set_operator(capi.Mat.from_scipy(sess, Mh))
    assert np.array_equal(solver.mult(b), x)
    solver.free()
    S.free()


# ------------------------------------------------------------------------------------------------------------------
# the kernels alone: the numeric-only product in every row-length bin (<= 64, <= 512, <= 4096 entries, longer rows in
# global memory) equals the two-pass product bit for bit; pe_smoother_update equals pe_smoother_create on the new values
@pytest.mark.parametrize("width", [8, 40, 300, 2500, 6000], ids=lambda w: "rowlen%d" % w)
def test_spgemm_numeric_bins(sess, width):
    import scipy.sparse as sp
    rng = np.random.default_rng(width)
    n, k = 64, 9000
    A = sp.random(n, k, density=min(1.0, 6.0 / k * max(1, width // 8)), random_state=rng, format="csr")
    B = sp.random(k, width, density=0.5, random_state=rng, format="csr")
    A2 = A.copy()
    A2.data = rng.standard_normal(A2.nnz)
    B2 = B.copy()
    B2.data = rng.standard_normal(B2.nnz)
    dA, dB, dA2, dB2 = [capi.Mat.from_scipy(sess, M) for M in (A, B, A2, B2)]
    Cm = capi.spgemm(sess, dA, dB)
    capi.spgemm_numeric(sess, dA2, dB2, Cm)
    want = capi.spgemm(sess, dA2, dB2)
    got, ref = Cm.to_scipy(), want.to_scipy()
    assert np.diff(ref.indptr).max() > width // 2
    assert np.array_equal(got.indptr, ref.indptr) and np.array_equal(got.indices, ref.indices)
    assert np.array_equal(got.data, ref.data)
    for m in (dA, dB, dA2, dB2, Cm, want):
        m.free()


@pytest.mark.parametrize("name,ordering,kernel,damping,omega,cheby",
                         [s for s in SMOOTHERS if s[0] != "Hypre Jacobi"],
                         ids=lambda v: str(v))
def test_smoother_update_equals_create(sess, hier, name, ordering, kernel, damping, omega, cheby):
    A1, marker = drivers.system_matrix(hier[0], 2, ESS)
    A2 = scaled(A1, marker, seed=3)
    b = np.random.default_rng(4).standard_normal(A1.shape[0])
    kw = dict(type=capi.SMOOTHER_TYPES[name], damping=damping, omega=omega, cheby_order=cheby,
              ordering=capi.GS_MULTICOLOR if ordering == "multicolor" else capi.GS_NATURAL)
    with with_sell(kernel):
        d1, d2 = capi.Mat.from_scipy(sess, A1), capi.Mat.from_scipy(sess, A2)
        su = capi.Smoother(sess, d1, **kw)
        su.update(d2)
        sf = capi.Smoother(sess, d2, **kw)
        out = []
        for sm in (su, sf):
            vb, vx = capi.Vec(sess, data=b), capi.Vec(sess, data=np.zeros_like(b))
            sm.apply(vb, vx, iterative_mode=False)
            out.append(vx.download())
        assert np.array_equal(su.l1(), sf.l1())
        assert su.eig() == sf.eig()
        su.free(); sf.free(); d1.free(); d2.free()
    assert np.array_equal(out[0], out[1])
