"""SetOperator on a built mixed (Darcy) solver (api.BlockSolver.set_blocks, pe_api_solver_set_operator_block): new values
for the blocks of [[M, Bt], [B, 0]] on the same patterns, as a new mobility or permeability sample brings them.  The
update must leave the solver in the state a fresh BuildSolver on the new blocks produces with the same sequence,
parameters, forms and boundary labels: every block Galerkin product, Schur complement and inner hierarchy is computed
numerically into the held patterns with the build's arithmetic, so preconditioner outputs, GMRES histories and level
blocks are compared bit for bit with a fresh build.  The hierarchy stays the one of the first sequence: M2 comes from
a second sequence on the same mesh with another coefficient.  A refused update changes nothing."""
import numpy as np
import pytest
import scipy.sparse as sp

import bench
from oracle import drivers
from parelag_b200 import api, capi

pytestmark = pytest.mark.gpu

DIMS, NLEV = (8, 8, 8), 3
NOESS = np.zeros((2, 6), dtype=np.int32)


@pytest.fixture(scope="module")
def sess():
    return api.session()


@pytest.fixture(scope="module")
def darcy(sess):
    """(S1, M1, M2, B, Bt): the hierarchy's sequence, its blocks and the H(div) mass block of a second sequence on the
    same mesh with a seeded coefficient 1/k per cell (host CSR copies; the device blocks are made per solver)"""
    S1 = api.Sequence.hex(DIMS, NLEV, jstart=2)
    M, B, Bt = S1.assemble_darcy(sess, 0)
    M1, Bh, Bth = M.to_scipy(), B.to_scipy(), Bt.to_scipy()
    kinv = 10.0 ** np.random.default_rng(3).uniform(-1.0, 1.0, DIMS[0] * DIMS[1] * DIMS[2])
    S2 = api.Sequence.hex(DIMS, NLEV, beta=kinv, jstart=2)
    M2d, B2d, Bt2d = S2.assemble_darcy(sess, 0)
    M2 = M2d.to_scipy()
    for m in (M, B, Bt, M2d, B2d, Bt2d):
        m.free()
    S2.free()
    assert np.array_equal(M1.indptr, M2.indptr) and np.array_equal(M1.indices, M2.indices)
    assert not np.array_equal(M1.data, M2.data)
    yield S1, M1, M2, Bh, Bth
    S1.free()


def dev(sess, blocks):
    return [[None if b is None else capi.Mat.from_scipy(sess, b) for b in row] for row in blocks]


def run_prec(sess, solver, rs, hierarchy):
    """preconditioner outputs on the same two device buffers, and how each call ran (blocked AMGe only)"""
    b, z = capi.Vec(sess, len(rs[0])), capi.Vec(sess, len(rs[0]))
    outs, modes = [], []
    for r in rs:
        b.upload(r)
        solver.prec_mult_device(b, z)
        outs.append(z.download())
        if hierarchy:
            modes.append(solver.replay_mode())
    b.free(); z.free()
    return outs, modes


def level_blocks(sess, solver):
    out = []
    for l in range(solver.num_levels()):
        for i in range(2):
            for j in range(2):
                m = solver.level_block(sess, l, i, j)
                out.append(None if m is None else m.to_scipy())
                if m is not None:
                    m.free()
    return out


def assert_same_blocks(got, want):
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(got, want)):
        assert (g is None) == (w is None), k
        if g is not None:
            assert np.array_equal(g.indptr, w.indptr) and np.array_equal(g.indices, w.indices), k
            assert np.array_equal(g.data, w.data), (k, np.abs(g.data - w.data).max())


def update_and_fresh(sess, S, xml, name, old, new, rs, b, hierarchy, ess=None):
    """(updated, fresh): outputs on rs, replay modes, GMRES (x, history), level blocks; the updated solver ran on rs
    before its update"""
    res = {}
    for which in ("upd", "fresh"):
        s = api.BlockSolver(xml, name, dev(sess, old if which == "upd" else new), S, 0, [2, 3], ess_attr=ess)
        if which == "upd":
            before, _ = run_prec(sess, s, rs, hierarchy)
            s.set_blocks(dev(sess, new))
        outs, modes = run_prec(sess, s, rs, hierarchy)
        x = s.mult(b)
        res[which] = dict(outs=outs, modes=modes, x=x, hist=s.history(), lev=level_blocks(sess, s) if hierarchy else None)
        s.free()
    assert not any(np.array_equal(p, q) for p, q in zip(before, res["upd"]["outs"]))
    return res["upd"], res["fresh"]


def assert_same_solver(upd, fresh):
    for o, f in zip(upd["outs"], fresh["outs"]):
        assert np.array_equal(o, f)
    assert upd["modes"] == fresh["modes"]
    assert np.array_equal(upd["hist"][0], fresh["hist"][0]) and upd["hist"][1:] == fresh["hist"][1:]
    assert np.array_equal(upd["x"], fresh["x"])
    if upd["lev"] is not None:
        assert_same_blocks(upd["lev"], fresh["lev"])


def rhs(n, k, seed):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal(n) for _ in range(k)], rng.standard_normal(n)


# ------------------------------------------------------------------------------------------------------------------
# 1: every block preconditioner of darcy_library_entries, with and without the blocked AMGe, and every S type
def _entry_cases():
    out = []
    for block, tri in (("Block Jacobi", None), ("Block GS", "Lower"), ("Block GS", "Upper"), ("Block LDU", None)):
        for amge in (True, False):
            for s_type in ("Diagonal", "AbsRowSum", "Mass"):
                out.append(pytest.param(block, tri, amge, s_type,
                                        id="%s%s-%s-%s" % (block.replace(" ", ""), tri or "", "amge" if amge else "single", s_type)))
    return out


@pytest.mark.parametrize("block,tri,amge,s_type", _entry_cases())
def test_update_matches_fresh_build(sess, darcy, block, tri, amge, s_type):
    S, M1, M2, B, Bt = darcy
    e = drivers.darcy_library_entries(block=block, amge=amge, s_type=s_type)
    if tri:
        e["Blk"][1]["Use triangle"] = tri
    rs, b = rhs(M1.shape[0] + B.shape[0], 4, seed=7)
    upd, fresh = update_and_fresh(sess, S, api.library_xml(e), "GMRES-AMGe-Blk", [[M1, Bt], [B, None]], [[M2, Bt], [B, None]],
                                  rs, b, hierarchy=amge)
    assert_same_solver(upd, fresh)


# the two solvers bench.py --config darcy / spe10 runs, natural and multicolour order
@pytest.mark.parametrize("ordering", ["natural", "multicolor"])
@pytest.mark.parametrize("which", ["library_darcy", "library_darcy_ldu"])
def test_bench_solvers_update_matches_fresh_build(sess, darcy, which, ordering):
    S, M1, M2, B, Bt = darcy
    ldu = which == "library_darcy_ldu"
    lib = getattr(bench, which)(ordering)
    name = "GMRES with Block LDU" if ldu else "GMRES with blocked AMGe"
    rs, b = rhs(M1.shape[0] + B.shape[0], 4, seed=8)
    upd, fresh = update_and_fresh(sess, S, api.library_xml(lib), name, [[M1, Bt], [B, None]], [[M2, Bt], [B, None]], rs, b,
                                  hierarchy=not ldu, ess=NOESS if ldu else None)
    assert_same_solver(upd, fresh)
    assert upd["hist"][2]


# ------------------------------------------------------------------------------------------------------------------
# 2: a non-zero A11 (S = A11 - A10 D^-1 A01: pe_spadd_numeric, off-diagonal R != P products), new values in all four
# blocks; and a new B of the same pattern in the Darcy system
def positive_scaled(A, seed):
    A = A.tocsr().copy()
    A.data = A.data * np.random.default_rng(seed).uniform(0.5, 2.0, A.nnz)
    return A


@pytest.mark.parametrize("block", ["Block GS", "Block Jacobi", "Block LDU"])
def test_nonzero_a11_unit_test_inputs(sess, block):
    """the inputs of the reference's block2x2 unit test (test_unit_block2x2_gpu.py), every block given new values"""
    M = sp.csr_matrix(np.array([[2., 1, 0, 0], [3, 4, 3, 0], [0, 3, 4, 3], [0, 0, 1, 2]]))
    Bt = sp.csr_matrix(np.array([[1., 0], [1, 1], [1, 1], [0, 1]]))
    B = sp.csr_matrix(np.array([[2., 1, 2, 0], [0, 2, 1, 2]]))
    Cm = sp.csr_matrix(np.array([[3., 0], [1, 3]]))
    old = [[M, Bt], [B, Cm]]
    new = [[positive_scaled(X, 10 + k) for k, X in enumerate(row)] for row in old]
    b, x0 = np.array([2., 1, 3, 1, 4, 1]), np.array([1., 2, 3, 4, 5, 6])
    if block == "Block LDU":
        p = {"A00_1 Inverse": "Gauss-Seidel", "A00_2 Inverse": "Gauss-Seidel", "A00_3 Inverse": "Gauss-Seidel",
             "S Inverse": "Gauss-Seidel", "S Type": "Diagonal"}
    else:
        p = {"A00 Inverse": "Gauss-Seidel", "A11 Inverse": "Gauss-Seidel", "S Type": "Diagonal"}
    xml = api.library_xml({"Gauss-Seidel": ("Hypre", {"Type": "Gauss-Seidel"}), "Blk": (block, p)})
    upd = api.BlockSolver(xml, "Blk", dev(sess, old), None, 0, [0, 0])
    x_old = upd.mult(b, x0=x0)
    upd.set_blocks(dev(sess, new))
    x_upd = upd.mult(b, x0=x0)
    upd.free()
    fresh = api.BlockSolver(xml, "Blk", dev(sess, new), None, 0, [0, 0])
    x_fresh = fresh.mult(b, x0=x0)
    fresh.free()
    assert not np.array_equal(x_old, x_upd)
    assert np.array_equal(x_upd, x_fresh)


@pytest.mark.parametrize("which", ["library_darcy", "library_darcy_ldu"])
def test_new_b_same_pattern(sess, darcy, which):
    """B' = diag(s) B with a seeded positive s, Bt' = Bt diag(s) (B'^T on Bt's pattern), and M2"""
    S, M1, M2, B, Bt = darcy
    s = np.random.default_rng(21).uniform(0.5, 2.0, B.shape[0])
    B2, Bt2 = B.copy(), Bt.copy()
    B2.data = B.data * s[np.repeat(np.arange(B.shape[0]), np.diff(B.indptr))]
    Bt2.data = Bt.data * s[Bt.indices]
    ldu = which == "library_darcy_ldu"
    name = "GMRES with Block LDU" if ldu else "GMRES with blocked AMGe"
    rs, b = rhs(M1.shape[0] + B.shape[0], 3, seed=22)
    upd, fresh = update_and_fresh(sess, S, api.library_xml(getattr(bench, which)("natural")), name, [[M1, Bt], [B, None]],
                                  [[M2, Bt2], [B2, None]], rs, b, hierarchy=not ldu, ess=NOESS if ldu else None)
    assert_same_solver(upd, fresh)


# ------------------------------------------------------------------------------------------------------------------
# 3: essential labels on the blocked hierarchy: the update fixes the recorded zero rows; a changed zero-row set of a
# coarse diagonal block is refused
ESS = np.array([np.ones(6, dtype=np.int32), np.zeros(6, dtype=np.int32)])


def zero_coarse_row(sess, S, M):
    """M with the rows and columns zeroed on the support of one column of the level-1 P of H(div) with ESS (one without
    essential rows): that coarse row of P^T M P becomes zero"""
    Pd = S.true_operator(sess, 0, "P", 2, ESS[0])
    P = Pd.to_scipy().tocsc()
    Pd.free()
    for c in range(P.shape[1]):
        rows = P.indices[P.indptr[c]:P.indptr[c + 1]][P.data[P.indptr[c]:P.indptr[c + 1]] != 0]
        if len(rows):
            break
    s = np.ones(M.shape[0])
    s[rows] = 0.0
    out = M.copy()
    r = np.repeat(np.arange(M.shape[0]), np.diff(M.indptr))
    out.data = M.data * s[r] * s[M.indices]
    return out


def test_essential_labels(sess, darcy):
    S, M1, M2, B, Bt = darcy
    xml = api.library_xml(bench.library_darcy("natural"))
    name = "GMRES with blocked AMGe"
    rs, b = rhs(M1.shape[0] + B.shape[0], 3, seed=31)
    upd, fresh = update_and_fresh(sess, S, xml, name, [[M1, Bt], [B, None]], [[M2, Bt], [B, None]], rs, b, hierarchy=True,
                                  ess=ESS)
    assert_same_solver(upd, fresh)
    s = api.BlockSolver(xml, name, dev(sess, [[M1, Bt], [B, None]]), S, 0, [2, 3], ess_attr=ESS)
    ref, _ = run_prec(sess, s, rs, True)
    with pytest.raises(capi.PEError, match="zero rows"):
        s.set_blocks(dev(sess, [[zero_coarse_row(sess, S, M2), Bt], [B, None]]))
    again, _ = run_prec(sess, s, rs, True)
    s.free()
    for o, r in zip(again, ref):
        assert np.array_equal(o, r)


# ------------------------------------------------------------------------------------------------------------------
# 4: M1 -> M2 -> M1 reproduces the solver built on M1
@pytest.mark.parametrize("which", ["library_darcy", "library_darcy_ldu"])
def test_round_trip(sess, darcy, which):
    S, M1, M2, B, Bt = darcy
    ldu = which == "library_darcy_ldu"
    name = "GMRES with Block LDU" if ldu else "GMRES with blocked AMGe"
    rs, _ = rhs(M1.shape[0] + B.shape[0], 3, seed=41)
    s = api.BlockSolver(api.library_xml(getattr(bench, which)("multicolor")), name, dev(sess, [[M1, Bt], [B, None]]), S, 0,
                        [2, 3], ess_attr=NOESS if ldu else None)
    ref, _ = run_prec(sess, s, rs, not ldu)
    lev_ref = None if ldu else level_blocks(sess, s)
    s.set_blocks(dev(sess, [[M2, Bt], [B, None]]))
    mid, _ = run_prec(sess, s, rs, not ldu)
    s.set_blocks(dev(sess, [[M1, Bt], [B, None]]))
    back, _ = run_prec(sess, s, rs, not ldu)
    if not ldu:
        assert_same_blocks(level_blocks(sess, s), lev_ref)
    s.free()
    assert not np.array_equal(mid[0], ref[0])
    for o, r in zip(back, ref):
        assert np.array_equal(o, r)


# ------------------------------------------------------------------------------------------------------------------
# 5: refusals name their reason and leave the solver computing what it computed
@pytest.mark.parametrize("which", ["library_darcy", "library_darcy_ldu"])
def test_refusals_change_nothing(sess, darcy, which):
    S, M1, M2, B, Bt = darcy
    ldu = which == "library_darcy_ldu"
    name = "GMRES with Block LDU" if ldu else "GMRES with blocked AMGe"
    nu, npr = M1.shape[0], B.shape[0]
    i = 0
    stored = set(M1.indices[M1.indptr[i]:M1.indptr[i + 1]])
    j = next(k for k in range(nu) if k not in stored)
    coo = M2.tocoo()
    extra = sp.csr_matrix((np.append(coo.data, 1e-3), (np.append(coo.row, i), np.append(coo.col, j))), shape=M2.shape)
    bigger = sp.block_diag([M2, sp.identity(1)]).tocsr()
    cases = [("zero block given a matrix", [[M2, Bt], [B, sp.identity(npr, format="csr")]], "zero"),
             ("non-zero block given NULL", [[M2, None], [B, None]], "zero"),
             ("extra entry", [[extra, Bt], [B, None]], "sparsity pattern"),
             ("block size", [[bigger, Bt], [B, None]], "size")]
    rs, _ = rhs(nu + npr, 3, seed=51)
    s = api.BlockSolver(api.library_xml(getattr(bench, which)("natural")), name, dev(sess, [[M1, Bt], [B, None]]), S, 0,
                        [2, 3], ess_attr=NOESS if ldu else None)
    ref, _ = run_prec(sess, s, rs, False)
    for what, blocks, reason in cases:
        with pytest.raises(capi.PEError, match=reason):
            s.set_blocks(dev(sess, blocks))
        again, _ = run_prec(sess, s, rs, False)
        for o, r in zip(again, ref):
            assert np.array_equal(o, r), what
    s.free()


# ------------------------------------------------------------------------------------------------------------------
# 6: the kernels alone against the ones they replace
def test_spadd_numeric_equals_spadd(sess):
    rng = np.random.default_rng(61)
    n, m = 300, 200
    A = sp.random(n, m, density=0.05, random_state=rng, format="csr")
    B = sp.random(n, m, density=0.05, random_state=rng, format="csr") + A     # shares some columns with A, not all
    B = sp.csr_matrix(B)
    A.sort_indices()
    rows_with_new = sum(len(set(B.indices[B.indptr[r]:B.indptr[r + 1]]) - set(A.indices[A.indptr[r]:A.indptr[r + 1]])) > 0
                        for r in range(n))
    assert rows_with_new > n // 2
    A2, B2 = A.copy(), B.copy()
    A2.data, B2.data = rng.standard_normal(A2.nnz), rng.standard_normal(B2.nnz)
    dA, dB, dA2, dB2 = [capi.Mat.from_scipy(sess, X) for X in (A, B, A2, B2)]
    Cm = capi.spadd(sess, 1.0, dA, -0.7, dB)
    capi.spadd_numeric(sess, 1.0, dA2, -0.7, dB2, Cm)
    want = capi.spadd(sess, 1.0, dA2, -0.7, dB2)
    got, ref = Cm.to_scipy(), want.to_scipy()
    assert np.array_equal(got.indptr, ref.indptr) and np.array_equal(got.indices, ref.indices)
    assert np.array_equal(got.data, ref.data)
    for x in (dA, dB, dA2, dB2, Cm, want):
        x.free()


@pytest.mark.parametrize("width", [8, 40, 300, 2500, 6000], ids=lambda w: "rowlen%d" % w)
def test_spgemm_numeric_scaled_bins(sess, width):
    """A diag(d)^-1 B into the held pattern equals copy (pe_spadd(1, B, 0, B)), pe_mat_scale_rows(copy, d, 1) and the
    two-pass product, in every row-length bin (<= 64, <= 512, <= 4096 entries, longer rows in global memory)"""
    rng = np.random.default_rng(width + 1)
    n, k = 64, 9000
    A = sp.random(n, k, density=min(1.0, 6.0 / k * max(1, width // 8)), random_state=rng, format="csr")
    B = sp.random(k, width, density=0.5, random_state=rng, format="csr")
    d = rng.uniform(0.1, 3.0, k) * rng.choice([-1.0, 1.0], k)
    dA, dB = capi.Mat.from_scipy(sess, A), capi.Mat.from_scipy(sess, B)
    vd = capi.Vec(sess, data=d)
    Cm = capi.spgemm(sess, dA, dB)
    capi.spgemm_numeric_scaled(sess, dA, vd, dB, Cm)
    copy = capi.spadd(sess, 1.0, dB, 0.0, dB)
    assert capi.lib().pe_mat_scale_rows(copy.h, vd.h, 1) == 0
    want = capi.spgemm(sess, dA, copy)
    got, ref = Cm.to_scipy(), want.to_scipy()
    assert np.diff(ref.indptr).max() > width // 2
    assert np.array_equal(got.indptr, ref.indptr) and np.array_equal(got.indices, ref.indices)
    assert np.array_equal(got.data, ref.data)
    for x in (dA, dB, Cm, copy, want):
        x.free()
    vd.free()


@pytest.mark.parametrize("cached", [False, True], ids=["transpose", "cached-transpose"])
def test_rap_numeric_rectangular_r(sess, cached):
    """R^T A P with a rectangular R != P (the off-diagonal blocks of a blocked level) equals pe_rap"""
    rng = np.random.default_rng(71)
    A = sp.random(400, 300, density=0.03, random_state=rng, format="csr")
    R = sp.random(400, 60, density=0.05, random_state=rng, format="csr")
    P = sp.random(300, 50, density=0.05, random_state=rng, format="csr")
    A2 = A.copy()
    A2.data = rng.standard_normal(A2.nnz)
    dA, dA2, dR, dP = [capi.Mat.from_scipy(sess, X) for X in (A, A2, R, P)]
    if cached:
        vx, vy = capi.Vec(sess, data=np.ones(400)), capi.Vec(sess, 60)
        dR.spmv_t(vx, vy)         # caches R^T on R
    Ac = capi.rap(sess, dA, dP, R=dR)
    assert Ac.info()[:2] == (60, 50)
    capi.rap_numeric(sess, dA2, dP, Ac, R=dR)
    want = capi.rap(sess, dA2, dP, R=dR)
    got, ref = Ac.to_scipy(), want.to_scipy()
    assert np.array_equal(got.indptr, ref.indptr) and np.array_equal(got.indices, ref.indices)
    assert np.array_equal(got.data, ref.data)
    for x in (dA, dA2, dR, dP, Ac, want):
        x.free()
