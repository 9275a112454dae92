"""Sign-encoded SELL SpMV and the zero-guess first colour of the multicolour SELL Gauss-Seidel sweep.

* A SpMV copy whose values are all -1, 0 or +1 (the discrete derivatives D of the fine de Rham sequence) stores int8
  codes instead of doubles.  The kernel decodes them to the same doubles and keeps the fma sequence, so y = D x is the
  sum of +-x_j in entry order, rounded after every term, bit for bit.  Any other value keeps the FP64 copy.
* A sweep from a zero initial guess does its first colour inside the renumbering pass: the rows of that colour only
  gather zeros.  The result must be bit-identical to the sweep that starts from an explicit zero vector, which runs the
  ordinary colour launch, and it takes one launch fewer.
* The H(curl) and H(div) V-cycles, whose Hiptmair smoothers use both, still match the oracle."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import amge, drivers
from parelag_b200 import api, capi

pytestmark = pytest.mark.gpu

ESS = np.ones(6, dtype=np.int32)


@pytest.fixture(scope="module")
def ctx():
    return api.session()


@pytest.fixture
def tuning():
    saved = {}

    def set_(key, value):
        saved.setdefault(key, capi.get_tuning(key))
        capi.set_tuning(key, value)
    yield set_
    for k, v in saved.items():
        capi.set_tuning(k, v)


def signed_matrix(m, n, per_row, seed, extra=None):
    """per_row entries per row with values -1, +1, 0.0 and -0.0, columns sorted; `extra` = value written into entry 7"""
    rng = np.random.default_rng(seed)
    rows = np.repeat(np.arange(m), per_row)
    cols = np.concatenate([np.sort(rng.choice(n, per_row, replace=False)) for _ in range(m)])
    vals = rng.choice(np.array([-1.0, 1.0, 1.0, -1.0, 0.0, -0.0]), m * per_row)
    if extra is not None:
        vals[7] = extra
    A = sp.csr_matrix((vals, (rows, cols)), shape=(m, n))
    A.data[:] = vals            # the constructor may drop the sign of -0.0 entries; keep every stored value as given
    return A


def entry_order_sum(A, x, y0=None):
    """row sums of a_ij x_j in stored order, rounded after every term; + y0 last (what fma(1, y0, acc) gives)"""
    y = np.zeros(A.shape[0])
    for i in range(A.shape[0]):
        acc = 0.0
        for k in range(A.indptr[i], A.indptr[i + 1]):
            acc = acc + A.data[k] * x[A.indices[k]]
        y[i] = acc if y0 is None else acc + y0[i]
    return y


def bits(v):
    return np.ascontiguousarray(v, dtype=np.float64).view(np.int64)


@pytest.mark.parametrize("per_row", [2, 4, 6, 11, 17])
def test_sign_coded_spmv_is_bit_exact(ctx, per_row):
    m, n = 3000, 2500
    A = signed_matrix(m, n, per_row, seed=per_row)
    rng = np.random.default_rng(1)
    x, y0 = rng.standard_normal(n), rng.standard_normal(m)
    dA = capi.Mat.from_scipy(ctx, A)
    dx, dy = capi.Vec(ctx, data=x), capi.Vec(ctx, m)
    capi.variant_counts(reset=True)
    dA.spmv(dx, dy, alpha=1.0, beta=0.0)
    assert np.array_equal(bits(dy.download()), bits(entry_order_sum(A, x)))
    dy.upload(y0)
    dA.spmv(dx, dy, alpha=1.0, beta=1.0)           # x += D x_aux of the Hiptmair smoother
    assert np.array_equal(bits(dy.download()), bits(entry_order_sum(A, x, y0)))
    counts = capi.variant_counts(reset=True)
    assert counts[capi.SPMV_SELL] == 2 * m and counts[capi.SPMV_SELL_SIGNS] == 2 * m
    for v in (dx, dy):
        v.free()


@pytest.mark.parametrize("value", [0.5, 2.0, -1.0000000000000002, 1e-300])
def test_other_values_keep_fp64(ctx, value):
    m, n = 3000, 2500
    A = signed_matrix(m, n, 4, seed=3, extra=value)
    x = np.random.default_rng(2).standard_normal(n)
    dA = capi.Mat.from_scipy(ctx, A)
    dx, dy = capi.Vec(ctx, data=x), capi.Vec(ctx, m)
    capi.variant_counts(reset=True)
    dA.spmv(dx, dy)
    counts = capi.variant_counts(reset=True)
    assert counts[capi.SPMV_SELL] == m and counts[capi.SPMV_SELL_SIGNS] == 0
    assert np.allclose(dy.download(), A @ x, rtol=0, atol=1e-14 * 4 * np.abs(x).max())
    for v in (dx, dy):
        v.free()


# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def hier():
    return amge.build_hierarchy((8, 8, 8), 3)[1]


def fp64_twin(A):
    """A with one more column whose only entry, 0.5 at the end of row 0, meets x = 0: the SELL copy of the twin keeps
    FP64 values, and its products are those of A (a +0 product added last leaves a row sum that is never -0 as it is)"""
    m, n = A.shape
    B = sp.hstack([A, sp.csr_matrix(([0.5], ([0], [0])), shape=(m, 1))], format="csr")
    B.sort_indices()
    return B


@pytest.mark.parametrize("form", [0, 1])
@pytest.mark.parametrize("transpose", [False, True], ids=["D", "DT"])
def test_fine_derivative_signs_match_fp64_and_separate_add(ctx, hier, form, transpose):
    """The discrete derivative D of the 8^3 fine sequence (form 0: the H1 gradient of the H(curl) Hiptmair smoother,
    form 1: the curl of the H(div) one) and its transpose: the sign-coded product equals the FP64 product of the same
    matrix bit for bit, and x += D x_aux in one pass (beta = 1) equals the product followed by the separate add."""
    D = sp.csr_matrix(hier[0].D[form])
    D = (D.T if transpose else D).tocsr()
    D.sort_indices()
    assert set(np.unique(D.data)) <= {-1.0, 0.0, 1.0}
    m, n = D.shape
    rng = np.random.default_rng(90 + form)
    x, y0 = rng.standard_normal(n), rng.standard_normal(m)
    dD, dT = capi.Mat.from_scipy(ctx, D), capi.Mat.from_scipy(ctx, fp64_twin(D))
    dx, dxt = capi.Vec(ctx, data=x), capi.Vec(ctx, data=np.append(x, 0.0))
    dy, dz, dw = capi.Vec(ctx, m), capi.Vec(ctx, m), capi.Vec(ctx, data=y0)
    capi.variant_counts(reset=True)
    dD.spmv(dx, dy)
    counts = capi.variant_counts(reset=True)
    assert counts[capi.SPMV_SELL_SIGNS] == m
    dT.spmv(dxt, dz)
    counts = capi.variant_counts(reset=True)
    assert counts[capi.SPMV_SELL] == m and counts[capi.SPMV_SELL_SIGNS] == 0
    assert np.array_equal(bits(dy.download()), bits(dz.download()))
    dw.axpby(1.0, dy, 1.0)                       # the separate add: w = D x + y0
    dz.upload(y0)
    dD.spmv(dx, dz, alpha=1.0, beta=1.0)         # the fused form: z = D x + z
    assert np.array_equal(bits(dz.download()), bits(dw.download()))
    for v in (dx, dxt, dy, dz, dw):
        v.free()


@pytest.mark.parametrize("form", [0, 1, 2])
@pytest.mark.parametrize("sweeps", [1, 2])
def test_zero_guess_first_colour_matches_the_colour_launch(ctx, hier, tuning, form, sweeps):
    """pe_smoother_apply from a zero guess vs from an uploaded zero vector (iterative mode): same bits, one launch
    fewer.  The comparison checks the row range of the first colour and the update expression of the folded pass."""
    tuning(capi.TUNE_SELL_MIN_ROWS, 0)          # the colour-ordered SELL sweep at this size
    tuning(capi.TUNE_FUSED_GS_MAX_MB, 0)        # one launch per colour (the fused sweep has its own zero-guess path)
    A, marker = drivers.system_matrix(hier[0], form, ESS)
    n = A.shape[0]
    rng = np.random.default_rng(40 + form)
    b = rng.standard_normal(n)
    b[marker] = 0.0
    dA = capi.Mat.from_scipy(ctx, A)
    s = capi.Smoother(ctx, dA, type=2, sweeps=sweeps, ordering=capi.GS_MULTICOLOR)
    _, starts = s.order()
    assert len(starts) > 2                       # several colours
    db, dx = capi.Vec(ctx, data=b), capi.Vec(ctx, n)
    out, launches = {}, {}
    for zero_guess in (True, False):
        dx.upload(np.zeros(n))
        l0 = ctx.launch_count()
        s.apply(db, dx, iterative_mode=not zero_guess)
        launches[zero_guess] = ctx.launch_count() - l0
        out[zero_guess] = dx.download()
    assert np.array_equal(bits(out[True]), bits(out[False]))
    assert launches[True] == launches[False] - 1
    assert np.any(out[True] != 0.0)
    s.free()
    for v in (db, dx):
        v.free()


# ---------------------------------------------------------------------------------------------------------------------
def _sequence(seqs):
    S = api.Sequence(4, len(seqs))
    for l, s in enumerate(seqs):
        for j in range(4):
            S.set_bdr_mask(l, j, drivers.bdr_mask(s.dof[j]))
            if j < 3:
                S.set_D(l, j, s.D[j])
            if l + 1 < len(seqs):
                S.set_P(l, j, s.P[j])
    return S


@pytest.mark.parametrize("form", [1, 2])
@pytest.mark.parametrize("mode", ["direct", "graph", "program"])
def test_hiptmair_vcycle_uses_sign_coded_d_and_matches_oracle(ctx, hier, tuning, form, mode):
    """Hiptmair V-cycle on the 8^3 H(curl) (form 1: D is the H1 gradient) and H(div) (form 2: D is the curl) systems,
    SELL family forced: the fine D and D^T are sign-coded, and the cycle matches the oracle in every execution mode."""
    tuning(capi.TUNE_SELL_MIN_ROWS, 0)
    tuning(capi.TUNE_FUSED_GS_MAX_MB, 0)
    A, marker = drivers.system_matrix(hier[0], form, ESS)
    n = A.shape[0]
    rng = np.random.default_rng(70 + form)
    rs = []
    for _ in range(4):
        r = rng.standard_normal(n)
        r[marker] = 0.0
        rs.append(r)
    e = drivers.library_entries(form, ordering="multicolor", smoother="L1 Gauss-Seidel", coarse_its=3, coarse_tol=1e-4,
                                hiptmair=True)
    e["AMGe"][1]["Use CUDA graph"] = mode != "direct"
    e["AMGe"][1]["Use persistent program"] = mode == "program"
    S = _sequence(hier)
    solver = api.Solver(api.library_xml(e), "PCG-AMGe", A, S, 0, form, ESS)
    b, z = capi.Vec(ctx, n), capi.Vec(ctx, n)
    capi.variant_counts(reset=True)
    outs = []
    for r in rs:
        b.upload(r)
        solver.prec_mult_device(b, z)
        outs.append(z.download())
    counts = capi.variant_counts(reset=True)
    assert counts[capi.SPMV_SELL_SIGNS] > 0
    H = drivers.amge_pcg_solver(hier, form, ESS, A, ordering="multicolor", hiptmair=True)
    for z_i, r in zip(outs, rs):
        zo = H.mult(r)
        assert np.linalg.norm(z_i - zo) <= 1e-11 * np.linalg.norm(zo)
    solver.free()
    S.free()
    for v in (b, z):
        v.free()
