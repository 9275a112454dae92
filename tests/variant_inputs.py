"""Inputs aimed at one side of each size threshold by which the host picks a kernel variant, and the exact references
the GPU results are checked against (tests/test_variants_gpu.py).

Each builder returns scipy CSR matrices together with the variant the host code will pick for them, computed here with
the same rule as the CUDA host code:
  - hash SpGEMM (pe_spgemm.cu run_bins): a row goes to the 128-, 1024- or 8192-slot shared table or to a global-memory
    table when its size is <= 64, <= 512, <= 4096 or larger; the symbolic pass sizes a row by the upper bound
    ub_i = sum_{k in A(i,:)} nnz(B(k,:)), the numeric pass by the exact nnz of row i of C;
  - single-rank SpMV (pe_spmv.cu pe_launch_spmv): SELL-32 when the padded SELL copy stores at most 1.25 x nnz entries,
    else the CTA streaming kernel when no row is longer than PE_STREAM_MAXROW = 512, else k_spmv<TPR>;
  - lanes per row of k_spmv, k_jacobi_update and k_gs_set (pe_core.cu pe_choose_tpr).
"""
import math

import numpy as np
import scipy.sparse as sp

SPGEMM_LIMITS = (64, 512, 4096)
SPGEMM_BINS = ("T128", "T1024", "T8192", "GMEM")
STREAM_MAXROW = 512
SELL_MAX_RATIO = 1.25
HASH_MULT = 2654435761
U = 2.0 ** -53


def _csr(indptr, indices, data, shape):
    return sp.csr_matrix((np.asarray(data, dtype=np.float64), np.asarray(indices, dtype=np.int32),
                          np.asarray(indptr, dtype=np.int32)), shape=shape)


def rows_to_csr(rows, ncols):
    """rows: list of (cols, vals) -> CSR with the entries in the given order (explicit zeros kept)"""
    indptr = np.zeros(len(rows) + 1, dtype=np.int64)
    for i, (c, _) in enumerate(rows):
        indptr[i + 1] = indptr[i] + len(c)
    J = np.concatenate([np.asarray(c, dtype=np.int64) for c, _ in rows]) if rows else np.zeros(0)
    A = np.concatenate([np.asarray(v, dtype=np.float64) for _, v in rows]) if rows else np.zeros(0)
    return _csr(indptr, J, A, (len(rows), ncols))


# ---------------------------------------------------------------------------------------------------------------------
# rules of the host code
# ---------------------------------------------------------------------------------------------------------------------
def spgemm_bin(size):
    """bin index of a row of the given size (k_bin_rows)"""
    size = np.asarray(size)
    return np.searchsorted(np.asarray(SPGEMM_LIMITS), size, side="left")


def spgemm_sizes(A, B):
    """(ub, nnz) per row of C = A B: the sizes the symbolic and the numeric pass bin on"""
    A, B = A.tocsr(), B.tocsr()
    rows = np.repeat(np.arange(A.shape[0]), np.diff(A.indptr))
    ub = np.bincount(rows, weights=np.diff(B.indptr)[A.indices], minlength=A.shape[0])
    return ub.astype(np.int64), np.diff(bool_product(A, B).indptr).astype(np.int64)


def spgemm_bin_counts(A, B):
    """expected pe_variant_counts of one C = A B: (symbolic counts, numeric counts) per bin.  The numeric pass does
    not run when C has no entries."""
    ub, nnz = spgemm_sizes(A, B)
    sym = np.bincount(spgemm_bin(ub), minlength=4) if A.shape[0] else np.zeros(4, dtype=np.int64)
    num = np.bincount(spgemm_bin(nnz), minlength=4) if nnz.sum() > 0 else np.zeros(4, dtype=np.int64)
    return sym, num


def choose_tpr(nnz, nrows):
    """pe_choose_tpr"""
    avg = nnz / nrows if nrows > 0 else 0.0
    t = 1
    while t < 32 and t * 1.5 < avg:
        t <<= 1
    return t


def sell_ratio(A):
    """stored entries of the SELL-32 copy (slices of 32 rows padded to their longest row, the last slice included)
    over nnz"""
    lens = np.diff(A.tocsr().indptr)
    pad = np.zeros(-len(lens) % 32, dtype=lens.dtype)
    w = np.concatenate([lens, pad]).reshape(-1, 32).max(axis=1)
    return 32.0 * w.sum() / A.nnz if A.nnz else math.inf


def spmv_path(A):
    """the kernel a single-rank SpMV with A takes: 'SELL', 'STREAM' or 'VECTOR'"""
    A = A.tocsr()
    if A.nnz > 0 and A.shape[0] > 0 and not (sell_ratio(A) > SELL_MAX_RATIO):
        return "SELL"
    if A.nnz > 0 and np.diff(A.indptr).max() <= STREAM_MAXROW:
        return "STREAM"
    return "VECTOR"


# ---------------------------------------------------------------------------------------------------------------------
# SpGEMM inputs
# ---------------------------------------------------------------------------------------------------------------------
def colliding_columns(table, count, first=0):
    """`count` column indices >= first that all hash to the last slot of a table of `table` slots:
    key * 2654435761 = table - 1 (mod table), i.e. key = (table - 1) * inverse (mod table), plus multiples of table"""
    k0 = ((table - 1) * pow(HASH_MULT, -1, table)) % table
    start = k0 + table * ((max(first - k0, 0) + table - 1) // table)
    cols = start + table * np.arange(count, dtype=np.int64)
    assert np.all((cols * HASH_MULT) % (2 ** 32) % table == table - 1)
    return cols


class _Builder:
    """rows of A on blocks of B rows: every A row references its own B rows, so row i of C is known by construction"""

    def __init__(self, rng, integer):
        self.rng, self.integer = rng, integer
        self.arows, self.brows = [], []

    def vals(self, n):
        if self.integer:
            v = self.rng.integers(1, 4, n) * self.rng.choice([-1, 1], n)
            return v.astype(np.float64)
        return self.rng.standard_normal(n) * 10.0 ** self.rng.uniform(-3, 3, n)

    def b_row(self, cols, vals=None):
        self.brows.append((np.asarray(cols, dtype=np.int64), self.vals(len(cols)) if vals is None else np.asarray(vals, float)))
        return len(self.brows) - 1

    def a_row(self, bidx, vals=None):
        self.arows.append((np.asarray(bidx, dtype=np.int64), self.vals(len(bidx)) if vals is None else np.asarray(vals, float)))

    def disjoint(self, total, parts, ncols):
        """A row with `parts` entries on B rows whose columns are disjoint: ub = nnz = total"""
        cols = self.rng.choice(ncols, total, replace=False)
        cuts = np.sort(self.rng.choice(np.arange(1, total), parts - 1, replace=False)) if parts > 1 else []
        self.a_row([self.b_row(c) for c in np.split(cols, cuts)])

    def shared(self, width, reps, ncols):
        """A row with `reps` entries on B rows with one common `width`-column pattern: ub = reps * width, nnz = width"""
        cols = self.rng.choice(ncols, width, replace=False)
        self.a_row([self.b_row(self.rng.permutation(cols)) for _ in range(reps)])

    def build(self, ncols):
        A = rows_to_csr(self.arows, len(self.brows))
        B = rows_to_csr(self.brows, ncols)
        return A, B


def spgemm_edges(integer, seed=0):
    """rows exactly at and just past every bin limit (ub = nnz = 64/65, 512/513, 4096/4097, built from 1-3 A entries on
    B rows with disjoint columns), rows whose ub and nnz fall into different bins (A entries on B rows with a common
    pattern), several bins in one matrix, empty A rows and A entries on empty B rows"""
    rng = np.random.default_rng(seed)
    b = _Builder(rng, integer)
    ncols = 9000
    for size in (1, 63, 64, 65, 511, 512, 513, 4095, 4096, 4097, 6000):
        for parts in (1, 2, 3):
            b.disjoint(size, min(parts, size), ncols)
    for width, reps in ((40, 2), (33, 2), (300, 2), (257, 2), (3000, 2), (50, 100), (8, 40), (400, 12)):
        b.shared(width, reps, ncols)
    b.a_row([])                                   # empty A row
    e = b.b_row([])
    b.a_row([e, e])                               # A entries on an empty B row: ub = 0
    b.a_row([e, b.b_row(rng.choice(ncols, 70, replace=False))])
    A, B = b.build(ncols)
    p = rng.permutation(A.shape[0])               # bins interleaved in row order
    return A[p], B


def spgemm_cancellation(seed=0):
    """small-integer rows with pairs +a, -a on B rows with the same pattern and values: those C entries are exactly 0.0
    and stay in the pattern; one bin each"""
    rng = np.random.default_rng(seed)
    b = _Builder(rng, True)
    ncols = 9000
    for width in (30, 200, 2000, 5000):
        cols = rng.choice(ncols, width, replace=False)
        v = b.vals(width)
        r0, r1 = b.b_row(cols, v), b.b_row(rng.permutation(cols), None)
        r2 = b.b_row(cols, v)
        a = float(rng.integers(1, 4))
        b.a_row([r0, r1, r2], [a, 1.0, -a])       # C row = B[r1]: the r0 / r2 products cancel exactly
        b.a_row([r0, r2], [a, -a])                # every entry exactly 0.0
    return b.build(ncols)


def spgemm_collisions(table, integer, seed=0):
    """one A row per fill level whose columns all hash to the last slot of the table the row is binned to: the
    linear probe wraps around the table end.  table: 128, 1024 or 8192 (the numeric row size fills half of it)"""
    rng = np.random.default_rng(seed)
    b = _Builder(rng, integer)
    full = table // 2
    cols = colliding_columns(table, full)
    ncols = int(cols[-1]) + 1
    for n, parts in ((full, 1), (full, 3), (full // 2 + 1, 2)):
        c = rng.permutation(cols[:n])
        cuts = np.sort(rng.choice(np.arange(1, n), parts - 1, replace=False)) if parts > 1 else []
        b.a_row([b.b_row(x) for x in np.split(c, cuts)])
    return b.build(ncols)


def spgemm_empty_product(seed=0):
    """every A entry points at an empty B row: nnz(C) = 0 (only the symbolic pass runs)"""
    A = _csr([0, 2, 2, 3], [0, 2, 1], [1.0, 2.0, 3.0], (3, 3))
    B = _csr([0, 0, 0, 0], [], [], (3, 7))
    return A, B


def rap_inputs(seed=0):
    """(A, P, R) for a Galerkin product whose two SpGEMMs use the 128-, 1024- and 8192-slot tables: a few long rows of P
    make long rows of A P and of R^T (A P); small integers (exact in FP64)"""
    rng = np.random.default_rng(seed)
    n = 600
    A = sp.random(n, n, density=0.01, random_state=rng, format="csr", data_rvs=lambda k: rng.integers(-3, 4, k).astype(float))
    A = (A + A.T + sp.identity(n) * 4.0).tocsr()
    cols = []
    for i in range(n):
        k = 300 if i % 97 == 0 else (40 if i % 7 == 0 else 1)     # a few long P rows
        cols.append(rng.choice(3000, k, replace=False))
    P = rows_to_csr([(c, rng.integers(1, 3, len(c)).astype(float)) for c in cols], 3000)
    R = rows_to_csr([(rng.choice(3000, 2, replace=False), [1.0, -1.0]) for _ in range(n)], 3000)
    return A, P, R


# ---------------------------------------------------------------------------------------------------------------------
# exact references
# ---------------------------------------------------------------------------------------------------------------------
def bool_product(A, B):
    """pattern of A B as a CSR of ones with sorted columns: the union of the B rows each A row references, whatever the
    values (so cancellation cannot remove an entry)"""
    A, B = A.tocsr(), B.tocsr()
    indptr, cols = [0], []
    for i in range(A.shape[0]):
        ks = A.indices[A.indptr[i]:A.indptr[i + 1]]
        c = np.unique(np.concatenate([B.indices[B.indptr[k]:B.indptr[k + 1]] for k in ks])) if len(ks) else np.zeros(0, np.int64)
        cols.append(c)
        indptr.append(indptr[-1] + len(c))
    J = np.concatenate(cols) if cols else np.zeros(0, np.int64)
    return _csr(indptr, J, np.ones(len(J)), (A.shape[0], B.shape[1]))


def two_product(a, b):
    """a*b = p + e exactly (Dekker / Veltkamp, no overflow in the inputs used here)"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    p = a * b
    f = 134217729.0                               # 2^27 + 1
    ta, tb = f * a, f * b
    ah, bh = ta - (ta - a), tb - (tb - b)
    al, bl = a - ah, b - bh
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def exact_product(A, B):
    """C = A B entry by entry, independently of any summation order: the pattern as a boolean product, and per entry the
    correctly rounded exact sum of the ROUNDED products fl(a_ik b_kj) (the kernels round every product before the shared
    -memory accumulation), the number of products k_ij and sum |a_ik b_kj|.  Returns (pattern CSR, values, k, abs_sum)
    in the pattern's order."""
    A, B = A.tocsr(), B.tocsr()
    C = bool_product(A, B)
    vals, kcnt, asum = np.zeros(C.nnz), np.zeros(C.nnz, dtype=np.int64), np.zeros(C.nnz)
    for i in range(A.shape[0]):
        lo, hi = C.indptr[i], C.indptr[i + 1]
        if lo == hi:
            continue
        terms = {}
        for q in range(A.indptr[i], A.indptr[i + 1]):
            k, a = A.indices[q], A.data[q]
            bl, bh = B.indptr[k], B.indptr[k + 1]
            prods = a * B.data[bl:bh]
            for j, pv in zip(B.indices[bl:bh].tolist(), prods.tolist()):
                terms.setdefault(j, []).append(pv)
        for p, j in enumerate(C.indices[lo:hi].tolist()):
            t = terms[j]
            vals[lo + p], kcnt[lo + p], asum[lo + p] = math.fsum(t), len(t), math.fsum(abs(x) for x in t)
    return C, vals, kcnt, asum


def exact_spmv(A, x, alpha=1.0, beta=0.0, y=None):
    """alpha A x + beta y per row as a correctly rounded exact sum (alpha a power of two, so alpha a_ik is exact), the
    number of terms (row length + 2: the products, the alpha scaling, the beta term) and the sum of |terms|"""
    A = A.tocsr()
    n = A.shape[0]
    p, e = two_product(alpha * A.data, x[A.indices])
    yb = np.zeros(n) if y is None or beta == 0.0 else y
    q, f = two_product(np.full(n, beta), yb)
    ref, asum = np.zeros(n), np.zeros(n)
    P, E, Pa = p.tolist(), e.tolist(), np.abs(p)
    for i in range(n):
        lo, hi = A.indptr[i], A.indptr[i + 1]
        ref[i] = math.fsum(P[lo:hi] + E[lo:hi] + [q[i], f[i]])
        asum[i] = float(Pa[lo:hi].sum()) + abs(q[i])
    return ref, np.diff(A.indptr) + 2, asum


# ---------------------------------------------------------------------------------------------------------------------
# SpMV inputs
# ---------------------------------------------------------------------------------------------------------------------
TPR_AVG = {1: 1.2, 2: 2.5, 4: 5.0, 8: 10.0, 16: 20.0, 32: 28.0}   # average row lengths inside each pe_choose_tpr interval


def _lengths(rng, n, total, maxlen):
    """n row lengths summing to total, spread unevenly (some empty rows), each <= maxlen"""
    base, extra = divmod(total, n)
    lens = np.full(n, base, dtype=np.int64)
    lens[rng.choice(n, extra, replace=False)] += 1
    for _ in range(n):                            # move entries between random rows
        i, j = rng.integers(0, n, 2)
        d = int(rng.integers(0, lens[i] + 1))
        d = min(d, maxlen - lens[j])
        lens[i] -= d
        lens[j] += d
    return lens


def matrix_from_lengths(rng, lens, ncols):
    rows = [(rng.choice(ncols, int(L), replace=False), rng.standard_normal(int(L))) for L in lens]
    return rows_to_csr(rows, ncols)


def spmv_vector_input(longest, tpr, seed=0):
    """one row of `longest` (> 512) entries, short other rows, average row length inside the interval of `tpr`: the
    lanes-per-row kernel k_spmv<tpr>"""
    rng = np.random.default_rng(seed)
    avg = TPR_AVG[tpr]
    n = int(math.ceil(2 * longest / avg)) + 37
    lens = _lengths(rng, n - 1, int(round(avg * n)) - longest, min(2 * int(avg) + 2, STREAM_MAXROW))
    lens = np.insert(lens, int(rng.integers(0, n)), longest)
    A = matrix_from_lengths(rng, lens, max(longest, 2 * n))
    assert spmv_path(A) == "VECTOR" and choose_tpr(A.nnz, A.shape[0]) == tpr
    return A


def spmv_stream_512(seed=0):
    """longest row exactly PE_STREAM_MAXROW = 512 entries, SELL rejected: the streaming kernel"""
    rng = np.random.default_rng(seed)
    lens = _lengths(rng, 999, 6000, 40)
    lens = np.insert(lens, 500, STREAM_MAXROW)
    A = matrix_from_lengths(rng, lens, 3000)
    assert spmv_path(A) == "STREAM"
    return A


def spmv_sell_padding(deficit, seed=0):
    """320 rows in 10 slices of width 10 with `deficit` entries removed: SELL stores 3200 entries for 3200 - deficit
    non-zeros.  deficit 630 -> ratio 1.246 (SELL), 640 -> exactly 1.25 (SELL), 650 -> 1.255 (streaming)"""
    rng = np.random.default_rng(seed)
    lens = np.full(320, 10, dtype=np.int64)
    lens[::32] = 10                                # every slice keeps one full row, so every slice is 10 wide
    cand = np.setdiff1d(np.arange(320), np.arange(0, 320, 32))
    for _ in range(deficit):
        i = rng.choice(cand[lens[cand] > 0])
        lens[i] -= 1
    return matrix_from_lengths(rng, lens, 500)


def spmv_edge_inputs(seed=0):
    """name -> matrix: nrows not a multiple of 32, empty rows, a single row (short and long), ncols >> nrows, an empty
    matrix"""
    rng = np.random.default_rng(seed)
    out = {}
    lens = rng.integers(0, 9, 1003)
    lens[rng.choice(1003, 150, replace=False)] = 0
    out["ragged_1003"] = matrix_from_lengths(rng, lens, 1003)
    out["single_row_short"] = matrix_from_lengths(rng, [10], 50)
    out["single_row_long"] = matrix_from_lengths(rng, [700], 5000)
    out["wide_5x100000"] = matrix_from_lengths(rng, [3000, 0, 17, 900, 1], 100000)
    out["all_empty_rows"] = _csr(np.zeros(40, dtype=np.int64), [], [], (39, 12))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# relaxation inputs (SPD, l1-Jacobi / natural-order Gauss-Seidel)
# ---------------------------------------------------------------------------------------------------------------------
def _lap1(n):
    return sp.diags([-np.ones(n - 1), 2 * np.ones(n), -np.ones(n - 1)], [-1, 0, 1])


def relax_inputs(seed=0):
    """tpr -> SPD matrix whose average row length selects that many lanes per row: a diagonal matrix with a few
    couplings (1), a 1-D (2), a 2-D (4) and a 3-D 7-point Laplacian (8), a 3-D 13-point stencil (16), a random
    diagonally dominant matrix with ~29 entries per row (32)"""
    rng = np.random.default_rng(seed)
    out = {}
    n = 1000
    i = rng.choice(n, 150, replace=False)
    j = (i + rng.integers(1, n, 150)) % n
    C = sp.coo_matrix((-rng.uniform(0.5, 1.0, 150), (i, j)), shape=(n, n)).tocsr()
    C = C + C.T
    out[1] = (C + sp.diags(rng.uniform(3.0, 5.0, n))).tocsr()
    out[2] = (_lap1(300) + sp.diags(np.full(300, 0.01))).tocsr()
    I10 = sp.identity(10)
    L10 = _lap1(10)
    out[8] = (sp.kron(sp.kron(L10, I10), I10) + sp.kron(sp.kron(I10, L10), I10) + sp.kron(sp.kron(I10, I10), L10)).tocsr()
    R = sp.random(600, 600, density=14 / 600, random_state=np.random.default_rng(seed + 1), format="csr")
    R.data[:] = -rng.uniform(0.1, 1.0, R.nnz)
    R = (R + R.T).tocsr()
    R.setdiag(0)
    R.eliminate_zeros()
    out[32] = (R + sp.diags(np.asarray(abs(R).sum(axis=1)).ravel() + 1.0)).tocsr()
    I = sp.identity(40)
    out[4] = (sp.kron(_lap1(40), I) + sp.kron(I, _lap1(40))).tocsr()
    m = 24
    t1 = sp.diags([np.ones(m - 1), np.ones(m - 1)], [-1, 1])
    t2 = sp.diags([np.ones(m - 2), np.ones(m - 2)], [-2, 2])
    Im = sp.identity(m)
    off = sum(sp.kron(sp.kron(a, b), c) for t in (t1, t2) for a, b, c in ((t, Im, Im), (Im, t, Im), (Im, Im, t)))
    out[16] = (sp.diags(np.full(m ** 3, 13.0)) - 0.5 * off).tocsr()
    for t, A in out.items():
        A.sort_indices()
        assert choose_tpr(A.nnz, A.shape[0]) == t, (t, A.nnz / A.shape[0])
    return out
