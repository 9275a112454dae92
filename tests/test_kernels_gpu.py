"""GPU parity tests of the solve-path kernels (through the C ABI) against the CPU
oracle on the same seeded inputs.  Integer outputs are bit-exact; FP64 tolerances
are stated per test."""
import numpy as np
import pytest
import scipy.sparse as sp

from parelag_b200 import capi
from oracle import solve as orc
from tests.util import laplace3d, random_spd, aggregation_P, sorted_csr

pytestmark = pytest.mark.gpu

RTOL_SPMV = 1e-13   # row sums are reduced in a different order than the sequential oracle


def _rel(a, b):
    return np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)


@pytest.mark.parametrize("maker", [lambda: laplace3d(9, 7, 5), lambda: random_spd(501, 0.05, 3),
                                   lambda: random_spd(64, 0.9, 4), lambda: laplace3d(40, 40, 40)])
def test_spmv_and_residual(ctx, maker):
    A = maker()
    n = A.shape[0]
    rng = np.random.default_rng(0)
    x, y0 = rng.standard_normal(n), rng.standard_normal(n)
    dA = capi.Mat.from_scipy(ctx, A)
    dx, dy = capi.Vec(ctx, data=x), capi.Vec(ctx, data=y0)
    dA.spmv(dx, dy, alpha=0.7, beta=-1.3)
    ref = orc.matvec(A, x, alpha=0.7, beta=-1.3, y=y0)
    assert _rel(dy.download(), ref) < RTOL_SPMV
    dA.spmv(dx, dy, alpha=1.0, beta=0.0)
    assert _rel(dy.download(), orc.matvec(A, x)) < RTOL_SPMV
    dr = capi.Vec(ctx, n)
    db = capi.Vec(ctx, data=y0)
    dA.residual(dx, db, dr)
    assert _rel(dr.download(), orc.matvec(A, x, alpha=-1.0, beta=1.0, y=y0)) < RTOL_SPMV
    for v in (dx, dy, dr, db):
        v.free()
    dA.free()


def test_spmv_rectangular_transpose_and_empty_rows(ctx):
    P = aggregation_P(7, 6, 5)
    # knock out some rows entirely (ragged / empty rows)
    P = P.tolil()
    P[3, :] = 0
    P[17, :] = 0
    P = P.tocsr()
    P.eliminate_zeros()
    rng = np.random.default_rng(1)
    xc, xf = rng.standard_normal(P.shape[1]), rng.standard_normal(P.shape[0])
    dP = capi.Mat.from_scipy(ctx, P)
    dxc, dxf = capi.Vec(ctx, data=xc), capi.Vec(ctx, data=xf)
    dyf, dyc = capi.Vec(ctx, P.shape[0]), capi.Vec(ctx, P.shape[1])
    dP.spmv(dxc, dyf)
    assert _rel(dyf.download(), orc.matvec(P, xc)) < RTOL_SPMV
    dP.spmv_t(dxf, dyc)
    assert _rel(dyc.download(), orc.matvec_t(P, xf)) < RTOL_SPMV
    # explicit transpose: pattern bit-exact (counting-sort order), values bit-exact
    T = dP.transpose().to_scipy()
    To = orc.transpose(P)
    assert np.array_equal(T.indptr, To.indptr) and np.array_equal(T.indices, To.indices)
    assert np.array_equal(T.data, To.data)


def test_vector_ops_and_dot(ctx):
    rng = np.random.default_rng(2)
    n = 100003
    x, y = rng.standard_normal(n), rng.standard_normal(n)
    dx, dy = capi.Vec(ctx, data=x), capi.Vec(ctx, data=y)
    d = dx.dot(dy)
    assert abs(d - float(x @ y)) <= 1e-12 * np.sqrt(float(x @ x) * float(y @ y))
    # deterministic: same bits on a second evaluation
    assert dx.dot(dy) == d
    dy.axpby(2.5, dx, -0.5)
    assert _rel(dy.download(), 2.5 * x - 0.5 * y) < 1e-15
    empty = capi.Vec(ctx, 0)
    assert empty.dot(empty) == 0.0


@pytest.mark.parametrize("stype", [1, 0, 5])
def test_jacobi_family(ctx, stype):
    A = random_spd(700, 0.02, 5)
    n = A.shape[0]
    rng = np.random.default_rng(3)
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    dA = capi.Mat.from_scipy(ctx, A)
    s = capi.Smoother(ctx, dA, type=stype, sweeps=2, damping=0.8)
    so = orc.Smoother(A, type=stype, sweeps=2, damping=0.8)
    assert _rel(s.l1(), so.l1) < 1e-15
    dx, db = capi.Vec(ctx, data=x0), capi.Vec(ctx, data=b)
    s.apply(db, dx, True)
    assert _rel(dx.download(), so.apply(b, x0, True)) < 1e-13
    s.apply(db, dx, False)
    assert _rel(dx.download(), so.apply(b, x0, False)) < 1e-13


@pytest.mark.parametrize("stype", [2, 4, 6])
@pytest.mark.parametrize("maker", [lambda: laplace3d(8, 9, 10), lambda: random_spd(400, 0.03, 7)])
def test_gauss_seidel_natural_order_is_hypre_order(ctx, stype, maker):
    """Level-scheduled GS == sequential natural-order sweep (hypre's order)."""
    A = maker()
    n = A.shape[0]
    rng = np.random.default_rng(4)
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    dA = capi.Mat.from_scipy(ctx, A)
    s = capi.Smoother(ctx, dA, type=stype, sweeps=1, ordering=capi.GS_NATURAL)
    so = orc.Smoother(A, type=stype, sweeps=1, order=None)
    # integer parity: the level of every row
    order, starts = s.order()
    lev = orc.natural_levels(A)
    glev = np.empty(n, dtype=np.int32)
    for c in range(len(starts) - 1):
        glev[order[starts[c]:starts[c + 1]]] = c
    assert np.array_equal(glev, lev)
    dx, db = capi.Vec(ctx, data=x0), capi.Vec(ctx, data=b)
    s.apply(db, dx, True)
    assert _rel(dx.download(), so.apply(b, x0, True)) < 1e-13


@pytest.fixture(params=["sell", "csr"])
def gs_kernel(request):
    """force the colour-ordered SELL-32 streaming kernel or the lanes-per-row CSR kernel"""
    old = capi.get_tuning(capi.TUNE_SELL_MIN_ROWS)
    capi.set_tuning(capi.TUNE_SELL_MIN_ROWS, 0 if request.param == "sell" else 1 << 30)
    yield request.param
    capi.set_tuning(capi.TUNE_SELL_MIN_ROWS, old)


@pytest.mark.parametrize("dims", [(11, 6, 7), (21, 20, 19)])
@pytest.mark.parametrize("stype", [2, 6])
@pytest.mark.parametrize("weights", [(1.0, 1.0), (0.9, 1.2)])
def test_gauss_seidel_multicolor(ctx, weights, gs_kernel, dims, stype):
    """stype 6 = hypre's "Gauss-Seidel" (division by the diagonal entry) with relaxation weight and omega"""
    A = laplace3d(*dims)
    n = A.shape[0]
    rng = np.random.default_rng(5)
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    dA = capi.Mat.from_scipy(ctx, A)
    s = capi.Smoother(ctx, dA, type=stype, sweeps=2, damping=weights[0], omega=weights[1],
                      ordering=capi.GS_MULTICOLOR)
    order, starts = s.order()
    oorder, ncol = orc.multicolor_order(A)
    assert len(starts) - 1 == ncol
    assert np.array_equal(order, oorder)          # integer parity: bit-exact colouring
    so = orc.Smoother(A, type=stype, sweeps=2, damping=weights[0], omega=weights[1], order=oorder)
    dx, db = capi.Vec(ctx, data=x0), capi.Vec(ctx, data=b)
    s.apply(db, dx, True)
    assert _rel(dx.download(), so.apply(b, x0, True)) < 1e-13


@pytest.mark.parametrize("ordering", ["multicolor", "natural"])
@pytest.mark.parametrize("maker", [lambda: laplace3d(21, 20, 19), lambda: _stencil27(11)])
def test_fused_sweep_kernel_is_bit_identical_to_per_colour_launches(ctx, gs_kernel, ordering, maker):
    """PE_TUNE_FUSED_GS_MAX_MB: the whole symmetric sweep (all colours / level sets, forward and backward, the SELL
    renumbering included) as ONE cooperative kernel with grid barriers -- same rows, same lanes, same summation order
    as one launch per colour, so the iterates are bit-identical; and both equal the oracle's sequential sweep."""
    if ordering == "natural" and gs_kernel == "sell":
        pytest.skip("natural-order level sets never take the SELL path; with the row threshold at 0 the per-set launches use the "
                    "streaming CSR kernel, whose row sums are accumulated in a different order than the lanes-per-row kernel")
    A = maker()
    n = A.shape[0]
    rng = np.random.default_rng(3)
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    dA = capi.Mat.from_scipy(ctx, A)
    old = capi.get_tuning(capi.TUNE_FUSED_GS_MAX_MB)
    out = {}
    try:
        for fused in (0, 24):
            capi.set_tuning(capi.TUNE_FUSED_GS_MAX_MB, fused)
            s = capi.Smoother(ctx, dA, type=2, sweeps=2, ordering=capi.GS_MULTICOLOR if ordering == "multicolor" else capi.GS_NATURAL)
            order, starts = s.order()
            for mode in (True, False):
                dx, db = capi.Vec(ctx, data=x0), capi.Vec(ctx, data=b)
                l0 = ctx.launch_count()
                s.apply(db, dx, mode)
                out[(fused, mode)] = (dx.download(), ctx.launch_count() - l0)
            s.free()
    finally:
        capi.set_tuning(capi.TUNE_FUSED_GS_MAX_MB, old)
    for mode in (True, False):
        assert np.array_equal(out[(0, mode)][0], out[(24, mode)][0])
        assert out[(24, mode)][1] == 2 and out[(0, mode)][1] > 2 * (len(starts) - 2)      # one launch per sweep vs per set
    so = orc.Smoother(A, type=2, sweeps=2, order=order if ordering == "multicolor" else None)
    assert _rel(out[(24, True)][0], so.apply(b, x0, True)) < 1e-13


def _stencil27(n):
    t = sp.diags([np.ones(n - 1), np.ones(n), np.ones(n - 1)], [-1, 0, 1])
    A = sp.kron(sp.kron(t, t), t).tocsr()
    A.data[:] = -1.0
    return (A + sp.diags(np.full(n ** 3, 27.0))).tocsr()


@pytest.mark.parametrize("maker", [lambda: laplace3d(21, 20, 19), lambda: _stencil27(13),
                                   lambda: sp.csr_matrix(aggregation_P(12, 10, 8))])
def test_sell_group_size_and_pdl_do_not_change_results(ctx, maker):
    """The SELL kernels' entry-group size (4/8/12, single-group or pipelined) and programmatic dependent
    launch are scheduling choices: SpMV and multicolour GS results are bit-identical across them and match
    the oracle (7-point: w<=7 single group of 8; 27-point: w=27 pipelined groups; P: w<=2)."""
    A = maker()
    square = A.shape[0] == A.shape[1]
    rng = np.random.default_rng(11)
    x, b = rng.standard_normal(A.shape[1]), rng.standard_normal(A.shape[0])
    old = [capi.get_tuning(k) for k in (capi.TUNE_SELL_MIN_ROWS, capi.TUNE_SELL_GROUP, capi.TUNE_PDL)]
    capi.set_tuning(capi.TUNE_SELL_MIN_ROWS, 0)
    results = []
    try:
        for group, pdl in [(0, 1), (0, 0), (4, 1), (8, 1), (12, 1), (12, 0)]:
            capi.set_tuning(capi.TUNE_SELL_GROUP, group)
            capi.set_tuning(capi.TUNE_PDL, pdl)
            dA = capi.Mat.from_scipy(ctx, A)
            dx, dy = capi.Vec(ctx, data=x), capi.Vec(ctx, A.shape[0])
            for _ in range(3):                      # back-to-back launches: the overlap PDL allows
                dA.spmv(dx, dy, alpha=1.0, beta=0.0)
            out = [dy.download()]
            if square:
                s = capi.Smoother(ctx, dA, type=2, sweeps=2, ordering=capi.GS_MULTICOLOR)
                du, db = capi.Vec(ctx, data=x), capi.Vec(ctx, data=b)
                s.apply(db, du, True)
                out.append(du.download())
            results.append(out)
    finally:
        for k, v in zip((capi.TUNE_SELL_MIN_ROWS, capi.TUNE_SELL_GROUP, capi.TUNE_PDL), old):
            capi.set_tuning(k, v)
    assert _rel(results[0][0], orc.matvec(A, x)) < RTOL_SPMV
    if square:
        oorder, _ = orc.multicolor_order(A)
        so = orc.Smoother(A, type=2, sweeps=2, order=oorder)
        assert _rel(results[0][1], so.apply(b, x, True)) < 1e-13
    for r in results[1:]:
        for a0, a1 in zip(results[0], r):
            assert np.array_equal(a0, a1)


@pytest.mark.parametrize("order", [1, 2, 3, 4])
def test_chebyshev(ctx, order):
    A = laplace3d(9, 9, 9)
    n = A.shape[0]
    rng = np.random.default_rng(6)
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    dA = capi.Mat.from_scipy(ctx, A)
    s = capi.Smoother(ctx, dA, type=16, sweeps=1, cheby_order=order, cheby_fraction=0.3)
    so = orc.Smoother(A, type=16, sweeps=1, cheby_order=order, cheby_fraction=0.3)
    mx, mn = s.eig()
    assert abs(mx - so.max_eig) < 1e-10 * so.max_eig and abs(mn - so.min_eig) < 1e-8 * so.max_eig
    dx, db = capi.Vec(ctx, data=x0), capi.Vec(ctx, data=b)
    s.apply(db, dx, True)
    assert _rel(dx.download(), so.apply(b, x0, True)) < 1e-11


@pytest.mark.parametrize("dims", [(6, 5, 4), (16, 16, 16), (3, 3, 3)])
def test_rap_pattern_bit_exact_values_1e12(ctx, dims):
    A = laplace3d(*dims)
    P = aggregation_P(*dims)
    dA, dP = capi.Mat.from_scipy(ctx, A), capi.Mat.from_scipy(ctx, P)
    Ac = capi.rap(ctx, dA, dP).to_scipy()
    Ao = orc.rap(A, P)
    assert np.array_equal(Ac.indptr, Ao.indptr)
    assert np.array_equal(Ac.indices, Ao.indices)      # sorted pattern, explicit zeros kept
    scale = np.max(np.abs(Ao.data))
    assert np.max(np.abs(Ac.data - Ao.data)) <= 1e-12 * scale


def test_spgemm_long_rows_use_bigger_tables(ctx):
    """rows with ~60 000 products and ~5 000 distinct columns: more than the 8192-slot shared table takes, so every
    row of both passes uses the global-memory table (the shared tables: tests/test_variants_gpu.py)."""
    rng = np.random.default_rng(8)
    A = sp.random(40, 3000, density=0.2, random_state=rng, format="csr")
    B = sp.random(3000, 5000, density=0.02, random_state=rng, format="csr")
    dA, dB = capi.Mat.from_scipy(ctx, A), capi.Mat.from_scipy(ctx, B)
    capi.variant_counts(reset=True)
    Cg = capi.spgemm(ctx, dA, dB).to_scipy()
    c = capi.variant_counts()
    assert list(c[[capi.SPGEMM_SYM_T128, capi.SPGEMM_SYM_T1024, capi.SPGEMM_SYM_T8192, capi.SPGEMM_SYM_GMEM]]) == [0, 0, 0, 40]
    assert list(c[[capi.SPGEMM_NUM_T128, capi.SPGEMM_NUM_T1024, capi.SPGEMM_NUM_T8192, capi.SPGEMM_NUM_GMEM]]) == [0, 0, 0, 40]
    Co = orc.spgemm(A, B)
    assert np.array_equal(Cg.indptr, Co.indptr) and np.array_equal(Cg.indices, Co.indices)
    assert np.max(np.abs(Cg.data - Co.data)) <= 1e-12 * np.max(np.abs(Co.data))


def test_fix_zero_rows_and_spadd(ctx):
    A = laplace3d(5, 5, 5).tolil()
    A[7, :] = 0
    A[7, 7] = 0.0
    A = A.tocsr()
    # keep an explicit zero row pattern: rebuild with stored zeros
    B = laplace3d(5, 5, 5)
    data = B.data.copy()
    lo, hi = B.indptr[7], B.indptr[8]
    data[lo:hi] = 0.0
    Z = sp.csr_matrix((data, B.indices, B.indptr), shape=B.shape)
    dZ = capi.Mat.from_scipy(ctx, Z)
    assert dZ.fix_zero_rows() == 1
    Zo, nf = orc.fix_zero_rows(Z)
    assert nf == 1
    G = dZ.to_scipy()
    assert np.array_equal(G.data, Zo.data)
    S = capi.spadd(ctx, 2.0, dZ, -3.0, capi.Mat.from_scipy(ctx, B)).to_scipy()
    assert abs(S - (2.0 * Zo - 3.0 * B)).max() < 1e-14


def test_hypre_extension_utilities(ctx):
    """src/hypreExtension on device matrices: delete-zeros, sign, identity/diagonal, norms, compare, RDP"""
    import scipy.sparse as sp
    rng = np.random.default_rng(21)
    A = sp.random(60, 45, density=0.15, random_state=3, format="csr")
    A.data = rng.standard_normal(A.nnz)
    A.data[::5] *= 1e-12
    dA = capi.Mat.from_scipy(ctx, A)
    nm = dA.norms()
    assert abs(nm["l1"] - abs(A).sum(axis=0).max()) < 1e-12 and abs(nm["linf"] - abs(A).sum(axis=1).max()) < 1e-12
    assert abs(nm["max"] - abs(A).max()) < 1e-14 and abs(nm["fro"] - np.sqrt((A.data ** 2).sum())) < 1e-12
    # compare: identical, perturbed, different shape
    dB = capi.Mat.from_scipy(ctx, A)
    assert dA.compare(dB, 1e-14) == 0
    B2 = A.copy(); B2.data[7] += 1e-3
    assert capi.Mat.from_scipy(ctx, B2).compare(dA, 1e-6) == 64
    assert capi.Mat.from_scipy(ctx, sp.csr_matrix(A[:50])).compare(dA, 1e-6) & (1 | 8 | 64)
    # delete zeros: hypre_CSRMatrixDeleteZeros deletes |a| <= tol (an entry equal to tol goes, tol = 0 removes the
    # stored zeros only)
    Z0 = A.copy(); Z0.data[3] = 0.0; Z0.data[11] = 0.0
    dZ0 = capi.Mat.from_scipy(ctx, Z0)
    dZ0.delete_zeros(0.0)
    G0 = dZ0.to_scipy()
    assert G0.nnz == A.nnz - 2 and abs(G0 - Z0).max() == 0
    A.data[1] = 1e-9                                      # exactly tol: deleted
    dA = capi.Mat.from_scipy(ctx, A)
    dA.delete_zeros(1e-9)
    Az = A.copy(); Az.data[np.abs(Az.data) <= 1e-9] = 0; Az.eliminate_zeros()
    G = dA.to_scipy()
    assert G.nnz == Az.nnz and abs(G - Az).max() == 0 and G[A.nonzero()[0][1], A.nonzero()[1][1]] == 0
    # sign
    dA.sign(1e-9)
    assert abs(dA.to_scipy() - Az.sign()).max() == 0
    # identity / diagonal
    d = rng.standard_normal(17)
    assert abs(capi.Mat.diagonal(ctx, 17).to_scipy() - sp.identity(17)).max() == 0
    assert abs(capi.Mat.diagonal(ctx, 17, capi.Vec(ctx, data=d)).to_scipy() - sp.diags(d)).max() == 0
    # R^T diag(d) P
    R = sp.random(30, 12, density=0.3, random_state=5, format="csr")
    P = sp.random(30, 9, density=0.3, random_state=6, format="csr")
    w = rng.standard_normal(30)
    out = capi.rdp(ctx, capi.Mat.from_scipy(ctx, R), capi.Vec(ctx, data=w), capi.Mat.from_scipy(ctx, P)).to_scipy()
    ref = (R.T @ sp.diags(w) @ P).tocsr()
    assert abs(out - ref).max() <= 1e-14 * max(abs(ref).max(), 1.0)
