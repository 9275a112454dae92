"""Every size-dispatched kernel variant against an exact reference, on inputs placed on either side of the threshold that
selects it (tests/variant_inputs.py).  Each test resets the process-wide variant counters (pe_variant_counts) and checks
that the variant it aims at really ran, on exactly the predicted number of rows, and that the other variants of the
family did not run where the input allows it."""
import numpy as np
import pytest

from oracle import amge
from oracle import solve as orc
from parelag_b200 import api, capi
from tests import variant_inputs as V
from tests.test_coarsen_gpu import compare_levels

pytestmark = pytest.mark.gpu

SPGEMM_SYM = [capi.SPGEMM_SYM_T128, capi.SPGEMM_SYM_T1024, capi.SPGEMM_SYM_T8192, capi.SPGEMM_SYM_GMEM]
SPGEMM_NUM = [capi.SPGEMM_NUM_T128, capi.SPGEMM_NUM_T1024, capi.SPGEMM_NUM_T8192, capi.SPGEMM_NUM_GMEM]
SPMV = {"SELL": capi.SPMV_SELL, "STREAM": capi.SPMV_STREAM, "VECTOR": capi.SPMV_VECTOR}
RELAX = {1: capi.RELAX_TPR_1, 2: capi.RELAX_TPR_2, 4: capi.RELAX_TPR_4, 8: capi.RELAX_TPR_8, 16: capi.RELAX_TPR_16,
         32: capi.RELAX_TPR_32}


def _named(counts, slots):
    return {capi.VARIANT_SLOTS[s]: int(counts[s]) for s in slots}


@pytest.fixture
def tuning():
    """set tuning keys inside a test; every key is restored afterwards"""
    saved = {}

    def set_(key, value):
        saved.setdefault(key, capi.get_tuning(key))
        capi.set_tuning(key, value)
    yield set_
    for k, v in saved.items():
        capi.set_tuning(k, v)


# ---------------------------------------------------------------------------------------------------------------------
# SpGEMM
# ---------------------------------------------------------------------------------------------------------------------
def _check_product(Cg, A, B, exact):
    """pattern equal to the boolean product (explicit zeros kept, ascending columns); values bit-exact (small integers)
    or within k_ij 2^-53 sum |a_ik b_kj| of the exact sum of the rounded products"""
    C, ref, k, asum = V.exact_product(A, B)
    assert Cg.shape == C.shape
    assert np.array_equal(Cg.indptr, C.indptr), "row lengths"
    assert np.array_equal(Cg.indices, C.indices), "columns"
    if exact:
        assert np.array_equal(Cg.data, ref)
    else:
        err = np.abs(Cg.data - ref)
        bound = k * V.U * asum
        bad = np.nonzero(err > bound)[0]
        assert bad.size == 0, (bad[:5], err[bad[:5]], bound[bad[:5]])


def _spgemm_and_check(ctx, A, B, exact):
    capi.variant_counts(reset=True)
    dA, dB = capi.Mat.from_scipy(ctx, A), capi.Mat.from_scipy(ctx, B)
    dC = capi.spgemm(ctx, dA, dB)
    counts = capi.variant_counts()
    Cg = dC.to_scipy()
    _check_product(Cg, A, B, exact)
    sym, num = V.spgemm_bin_counts(A, B)
    assert _named(counts, SPGEMM_SYM) == _named(dict(zip(SPGEMM_SYM, sym)), SPGEMM_SYM)
    assert _named(counts, SPGEMM_NUM) == _named(dict(zip(SPGEMM_NUM, num)), SPGEMM_NUM)
    for m in (dA, dB, dC):
        m.free()
    return sym, num


@pytest.mark.parametrize("exact", [True, False], ids=["small_integers", "random_fp64"])
def test_spgemm_rows_at_every_bin_limit(ctx, exact):
    """ub = nnz at 64/65, 512/513, 4096/4097 and beyond, rows whose ub and nnz fall into different bins, empty rows:
    every table of both passes runs in one product"""
    A, B = V.spgemm_edges(exact, seed=1)
    sym, num = _spgemm_and_check(ctx, A, B, exact)
    assert np.all(sym > 0) and np.all(num > 0)


def test_spgemm_cancellation_keeps_exact_zeros(ctx):
    """+a and -a products of equal values: those entries are exactly 0.0 and stay in the pattern (as hypre keeps them)"""
    A, B = V.spgemm_cancellation(seed=2)
    _, ref, _, _ = V.exact_product(A, B)
    assert np.count_nonzero(ref == 0.0) == 30 + 200 + 2000 + 5000      # the device result equals ref bit for bit
    _spgemm_and_check(ctx, A, B, True)


@pytest.mark.parametrize("table", [128, 1024, 8192])
@pytest.mark.parametrize("exact", [True, False], ids=["small_integers", "random_fp64"])
def test_spgemm_hash_collisions_wrap_around(ctx, table, exact):
    """every column hashes to the last slot of the table its row is binned to: linear probing wraps around the end of
    the table, at half fill (the most the host lets into a table) and below"""
    A, B = V.spgemm_collisions(table, exact, seed=3)
    sym, num = _spgemm_and_check(ctx, A, B, exact)
    b = {128: 0, 1024: 1, 8192: 2}[table]
    assert sym[b] == num[b] == A.shape[0]


def test_spgemm_empty_inputs(ctx):
    """A entries on empty B rows (nnz(C) = 0: only the symbolic pass runs), and A with 0 rows (nothing runs)"""
    A, B = V.spgemm_empty_product()
    sym, num = _spgemm_and_check(ctx, A, B, True)
    assert sym[0] == 3 and num.sum() == 0
    A0 = V._csr([0], [], [], (0, 4))
    B0 = V._csr([0, 1, 1, 3, 3], [2, 0, 4], [1.0, 2.0, 3.0], (4, 6))
    sym, num = _spgemm_and_check(ctx, A0, B0, True)
    assert sym.sum() == 0 and num.sum() == 0


@pytest.mark.parametrize("with_R", [False, True])
def test_rap_exact_over_the_shared_tables(ctx, with_R):
    """P^T A P and R^T A P of small integers: bit-exact against the exact integer product, the counters of both SpGEMMs
    as the binning rule predicts"""
    A, P, R = V.rap_inputs(seed=4)
    C1, v1, _, _ = V.exact_product(A, P)
    AP = V._csr(C1.indptr, C1.indices, v1, C1.shape)
    Rt = (R if with_R else P).T.tocsr()
    C2, v2, _, _ = V.exact_product(Rt, AP)
    capi.variant_counts(reset=True)
    dA, dP = capi.Mat.from_scipy(ctx, A), capi.Mat.from_scipy(ctx, P)
    dR = capi.Mat.from_scipy(ctx, R) if with_R else None
    Ac = capi.rap(ctx, dA, dP, dR).to_scipy()
    counts = capi.variant_counts()
    assert np.array_equal(Ac.indptr, C2.indptr) and np.array_equal(Ac.indices, C2.indices)
    assert np.array_equal(Ac.data, v2)
    s1, n1 = V.spgemm_bin_counts(A, P)
    s2, n2 = V.spgemm_bin_counts(Rt, AP)
    assert list(counts[SPGEMM_SYM]) == list(s1 + s2) and list(counts[SPGEMM_NUM]) == list(n1 + n2)
    assert np.all(counts[SPGEMM_NUM[:3]] > 0)


# ---------------------------------------------------------------------------------------------------------------------
# SpMV
# ---------------------------------------------------------------------------------------------------------------------
def _spmv_checks(ctx, A, path, seed=0):
    """y = A x, y = 2 A x - 1.3 y0, r = b - A x and y = A^T x against exact row sums; the forward products take `path`"""
    rng = np.random.default_rng(seed)
    m, n = A.shape
    x, y0, xt = rng.standard_normal(n), rng.standard_normal(m), rng.standard_normal(m)
    dA = capi.Mat.from_scipy(ctx, A)
    dx, dy, dr, db = capi.Vec(ctx, data=x), capi.Vec(ctx, m), capi.Vec(ctx, m), capi.Vec(ctx, data=y0)
    dxt, dyt = capi.Vec(ctx, data=xt), capi.Vec(ctx, n)
    capi.variant_counts(reset=True)
    cases = []
    dA.spmv(dx, dy, alpha=1.0, beta=0.0)
    cases.append((dy.download(), V.exact_spmv(A, x)))
    dy.upload(y0)
    dA.spmv(dx, dy, alpha=2.0, beta=-1.3)
    cases.append((dy.download(), V.exact_spmv(A, x, 2.0, -1.3, y0)))
    dA.residual(dx, db, dr)
    cases.append((dr.download(), V.exact_spmv(A, x, -1.0, 1.0, y0)))
    counts = capi.variant_counts(reset=True)
    assert _named(counts, SPMV.values()) == {capi.VARIANT_SLOTS[s]: (3 * m if k == path else 0) for k, s in SPMV.items()}
    dA.spmv_t(dxt, dyt, alpha=-0.5, beta=0.0)
    assert capi.variant_counts()[SPMV[V.spmv_path(A.T.tocsr())]] == n
    cases.append((dyt.download(), V.exact_spmv(A.T.tocsr(), xt, -0.5)))
    for got, (ref, k, asum) in cases:
        err, bound = np.abs(got - ref), k * V.U * asum
        bad = np.nonzero(err > bound)[0]
        assert bad.size == 0, (bad[:5], err[bad[:5]], bound[bad[:5]])
    for v in (dx, dy, dr, db, dxt, dyt):
        v.free()
    dA.free()


@pytest.mark.parametrize("tpr", [1, 2, 4, 8, 16, 32])
@pytest.mark.parametrize("longest", [513, 2000, 20000])
def test_spmv_lanes_per_row_every_tpr(ctx, longest, tpr):
    """one row longer than the streaming kernel admits: k_spmv<TPR> with the TPR the average row length selects"""
    A = V.spmv_vector_input(longest, tpr, seed=longest + tpr)
    _spmv_checks(ctx, A, "VECTOR", seed=tpr)


@pytest.mark.parametrize("name", ["stream_512", "sell_1.246", "sell_1.25", "stream_1.255"])
def test_spmv_threshold_neighbours(ctx, name):
    """longest row exactly 512 (streaming), SELL padding just under, at and just over 25 %"""
    A = V.spmv_stream_512() if name == "stream_512" else V.spmv_sell_padding({"sell_1.246": 630, "sell_1.25": 640,
                                                                              "stream_1.255": 650}[name])
    path = name.split("_")[0].upper()
    assert V.spmv_path(A) == path
    _spmv_checks(ctx, A, path)


@pytest.mark.parametrize("name", sorted(V.spmv_edge_inputs()))
def test_spmv_shape_edges(ctx, name):
    """nrows not a multiple of 32, empty rows, one row, ncols >> nrows, no entries at all"""
    A = V.spmv_edge_inputs()[name]
    _spmv_checks(ctx, A, V.spmv_path(A))


# ---------------------------------------------------------------------------------------------------------------------
# relaxation
# ---------------------------------------------------------------------------------------------------------------------
def _rel(a, b):
    return np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)


@pytest.mark.parametrize("tpr", [1, 2, 4, 8, 16, 32])
@pytest.mark.parametrize("stype,weights", [(1, (0.8, 1.0)), (2, (1.0, 1.0)), (6, (1.0, 1.0)), (6, (0.9, 1.2)),
                                           (2, (0.9, 1.2))])
def test_relaxation_lanes_per_row(ctx, tpr, stype, weights):
    """l1-Jacobi (k_jacobi_update<TPR>) and natural-order Gauss-Seidel (k_gs_set<TPR, GENERAL>) against the oracle's
    sequential sweep; natural order fixes the operand values of every row"""
    A = V.relax_inputs()[tpr]
    n = A.shape[0]
    rng = np.random.default_rng(tpr)
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    dA = capi.Mat.from_scipy(ctx, A)
    s = capi.Smoother(ctx, dA, type=stype, sweeps=2, damping=weights[0], omega=weights[1], ordering=capi.GS_NATURAL)
    so = orc.Smoother(A, type=stype, sweeps=2, damping=weights[0], omega=weights[1], order=None)
    dx, db = capi.Vec(ctx, data=x0), capi.Vec(ctx, data=b)
    capi.variant_counts(reset=True)
    s.apply(db, dx, True)
    counts = capi.variant_counts()
    assert _rel(dx.download(), so.apply(b, x0, True)) < 1e-13
    per_sweep = n if stype == 1 else 2 * n          # Gauss-Seidel: forward and backward pass
    assert _named(counts, RELAX.values()) == {capi.VARIANT_SLOTS[v]: (2 * per_sweep if t == tpr else 0) for t, v in RELAX.items()}
    s.free()
    dA.free()


# ---------------------------------------------------------------------------------------------------------------------
# batched local solves of Coarsen()
# ---------------------------------------------------------------------------------------------------------------------
LOCAL = [capi.TRACES_SMEM, capi.TRACES_GMEM, capi.EXT_SMEM, capi.EXT_GMEM]


def _outputs(S, nlev, jstart):
    """every operator and table Coarsen() produced, as arrays"""
    out = {}
    for l in range(nlev):
        for j in range(jstart, 4):
            mats = {}
            if l + 1 < nlev:
                mats["P"] = S.get_csr(l, "P", j)
            if j < 3:
                mats["D"] = S.get_csr(l, "D", j)
            if l > 0:
                for cd in range(4 - j):
                    mats["Me%d" % cd] = S.get_csr(l, "Me", j, cd)
                    mats["ED%d" % cd] = S.get_csr(l, "ED", j, cd)
                out[(l, j, "targets")] = S.get_targets(l, j)
                out[(l, j, "bdr")] = S.get_bdr_mask(l, j)
            for name, M in mats.items():
                out[(l, j, name)] = (M.shape, M.indptr.copy(), M.indices.copy(), M.data.copy())
    return out


def _assert_bit_identical(a, b):
    assert a.keys() == b.keys()
    for k in a:
        x, y = a[k], b[k]
        if isinstance(x, tuple):
            assert x[0] == y[0] and all(np.array_equal(p, q) for p, q in zip(x[1:], y[1:])), k
        else:
            assert x.shape == y.shape and np.array_equal(x, y), k


def _run(make, tuning, smem_bytes):
    tuning(capi.TUNE_LOCAL_SMEM_BYTES, smem_bytes)
    capi.variant_counts(reset=True)
    S = make()
    return S, capi.variant_counts()


def _cases():
    rng = np.random.default_rng(7)
    aniso = dict(dims=(4, 4, 4), nlev=2, kw=dict(L=(1.0, 2.0, 0.5), alpha=rng.uniform(0.5, 2.0, 64),
                                                beta=10.0 ** rng.uniform(-2, 2, 64)), jstart=0, tol=1e-10, null_tol=None)
    rng = np.random.default_rng(11)
    deformed = dict(dims=(4, 4, 4), nlev=3, kw=dict(alpha=rng.uniform(0.5, 2.0, 64), beta=10.0 ** rng.uniform(-1, 1, 64)),
                    jstart=1, tol=1e-10, null_tol=1e-7, deform=True)
    return {"uniform_8": dict(dims=(8, 8, 8), nlev=3, kw={}, jstart=0, tol=1e-12, null_tol=None),
            "anisotropic_nullspace": aniso, "deformed_hcurl_dense_trace": deformed}


def _setup(case):
    c = _cases()[case]
    dims, nlev, kw, jstart = c["dims"], c["nlev"], dict(c["kw"]), c["jstart"]
    deform = amge.weak_scaling_deformation if c.get("deform") else None
    mesh, seqs = amge.build_hierarchy(dims, nlev, jstart=jstart, deform=deform, **kw)
    if deform:
        kw = dict(alpha=kw["alpha"], beta=kw["beta"], coords=mesh.vertex_coords())

    def make():
        return api.Sequence.hex(dims, nlev, jstart=jstart, **kw)
    return c, seqs, make


@pytest.mark.parametrize("case", ["uniform_8", "anisotropic_nullspace", "deformed_hcurl_dense_trace"])
def test_local_solves_global_workspace_is_bit_identical(tuning, case):
    """PE_TUNE_LOCAL_SMEM_BYTES = 1 sends every agglomerate to k_traces_gmem / k_extension_gmem: every output of Coarsen()
    is bit-identical to the shared-memory run, and matches the oracle."""
    api.session()
    c, seqs, make = _setup(case)
    nlev, jstart = c["nlev"], c["jstart"]
    S0, c0 = _run(make, tuning, 0)
    ref = _outputs(S0, nlev, jstart)
    S0.free()
    assert c0[capi.TRACES_SMEM] > 0 and c0[capi.EXT_SMEM] > 0 and c0[capi.TRACES_GMEM] == 0
    if case != "deformed_hcurl_dense_trace":
        assert c0[capi.EXT_GMEM] == 0
    S1, c1 = _run(make, tuning, 1)
    assert c1[capi.TRACES_SMEM] == 0 and c1[capi.EXT_SMEM] == 0 and c1[capi.EXT_SPLIT_SMEM] == 0
    assert c1[capi.TRACES_GMEM] == c0[capi.TRACES_SMEM] + c0[capi.TRACES_GMEM]
    assert c1[capi.EXT_GMEM] == c0[capi.EXT_SMEM] + c0[capi.EXT_GMEM]
    _assert_bit_identical(_outputs(S1, nlev, jstart), ref)
    compare_levels(S1, seqs, tol=c["tol"], null_tol=c["null_tol"])
    S1.free()


LIMIT_MAX = 220 * 1024      # the larger built-in limit: the knob is clamped to it


def test_local_solves_split_batch_is_bit_identical(tuning):
    """A knob value between the workspace sizes of the agglomerates of ONE extension batch splits that batch: the
    agglomerates that fit run in the listed k_extension launch (carve-up from the bounds of that subset), the others
    in k_extension_gmem.  EXT_SPLIT_SMEM counts the listed launch on its own.  The knob is searched by interval
    subdivision over the values where the shared-memory share changes; every output must be bit-identical to the
    default run and to the run with every agglomerate on the global-workspace kernels.  The deformed H(curl) case has
    agglomerates of different workspace within one batch (NullSpace dofs on some entities only); in the uniform and the
    anisotropic cases the agglomerates of a batch have equal workspace, so no knob value splits a batch there."""
    api.session()
    c, seqs, make = _setup("deformed_hcurl_dense_trace")
    nlev, jstart = c["nlev"], c["jstart"]
    S0, _ = _run(make, tuning, 0)
    ref = _outputs(S0, nlev, jstart)
    S0.free()
    S1, c1 = _run(make, tuning, 1)
    all_gmem = _outputs(S1, nlev, jstart)
    S1.free()
    _assert_bit_identical(all_gmem, ref)
    seen = {1: c1}

    def smem_share(v):
        S, cv = _run(make, tuning, v)
        seen[v] = cv
        if cv[capi.EXT_SPLIT_SMEM] > 0:
            return S
        S.free()
        return None
    found = smem_share(LIMIT_MAX)
    todo = [(1, LIMIT_MAX)]
    while found is None and todo and len(seen) < 80:
        lo, hi = todo.pop()
        if hi - lo < 2 or seen[lo][capi.EXT_SMEM] == seen[hi][capi.EXT_SMEM]:
            continue
        mid = (lo + hi) // 2
        found = smem_share(mid)
        todo += [(lo, mid), (mid, hi)]
    assert found is not None, ("no knob value splits an extension batch", {
        v: tuple(int(cv[k]) for k in (capi.EXT_SMEM, capi.EXT_GMEM, capi.EXT_SPLIT_SMEM)) for v, cv in sorted(seen.items())})
    v = max(k for k in seen if seen[k][capi.EXT_SPLIT_SMEM] > 0)
    cv = seen[v]
    assert 0 < cv[capi.EXT_SPLIT_SMEM] <= cv[capi.EXT_SMEM] and cv[capi.EXT_GMEM] > 0
    split = _outputs(found, nlev, jstart)
    found.free()
    _assert_bit_identical(split, ref)
    _assert_bit_identical(split, all_gmem)


def test_local_solves_grid_stride_loop_reuses_workspace(tuning):
    """20^3, 2 levels, every agglomerate on the global-workspace kernels: single launches with more agglomerated
    entities than CTAs (148 x 16 traces, 148 x 4 extension), so each CTA's slab serves several agglomerates in turn
    (TRACES_GMEM_REUSE / EXT_GMEM_REUSE count those later turns).  No state may carry over: every output bit-identical to
    the shared-memory run."""
    api.session()
    dims, nlev = (20, 20, 20), 2

    def make():
        return api.Sequence.hex(dims, nlev)
    S0, c0 = _run(make, tuning, 0)
    ref = _outputs(S0, nlev, 0)
    S0.free()
    S1, c1 = _run(make, tuning, 1)
    assert c1[capi.TRACES_GMEM_REUSE] > 0 and c1[capi.EXT_GMEM_REUSE] > 0
    assert c1[capi.TRACES_SMEM] == 0 and c1[capi.EXT_SMEM] == 0 and c0[capi.TRACES_GMEM] == 0 and c0[capi.EXT_GMEM] == 0
    assert c0[capi.TRACES_GMEM_REUSE] == 0 and c0[capi.EXT_GMEM_REUSE] == 0
    _assert_bit_identical(_outputs(S1, nlev, 0), ref)
    S1.free()
