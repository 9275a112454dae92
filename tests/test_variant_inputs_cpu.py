"""The inputs of tests/test_variants_gpu.py land on the intended side of every dispatch threshold (checked here with the
host code's rules, no GPU), and the exact references they are compared with are exact."""
import math
from fractions import Fraction

import numpy as np
import pytest

from tests import variant_inputs as V


def test_spgemm_edge_rows_sit_at_the_bin_limits():
    A, B = V.spgemm_edges(True, seed=1)
    ub, nnz = V.spgemm_sizes(A, B)
    for size in (64, 65, 512, 513, 4096, 4097):
        assert np.any((ub == size) & (nnz == size)), size
    assert np.any(V.spgemm_bin(ub) != V.spgemm_bin(nnz))          # ub and nnz in different bins
    assert np.any((V.spgemm_bin(ub) == 3) & (V.spgemm_bin(nnz) == 0))
    assert np.any(np.diff(A.indptr) == 0) and np.any((ub == 0) & (np.diff(A.indptr) > 0))
    sym, num = V.spgemm_bin_counts(A, B)
    assert np.all(sym > 0) and np.all(num > 0)
    assert list(V.spgemm_bin([0, 64, 65, 512, 513, 4096, 4097])) == [0, 0, 1, 1, 2, 2, 3]


@pytest.mark.parametrize("table", [128, 1024, 8192])
def test_collision_columns_hash_to_the_last_slot(table):
    cols = V.colliding_columns(table, table // 2)
    assert len(set(cols.tolist())) == table // 2
    slots = (cols.astype(object) * 2654435761) % 2 ** 32 % table         # the device's hash in exact integers
    assert set(slots.tolist()) == {table - 1}
    A, B = V.spgemm_collisions(table, True)
    ub, nnz = V.spgemm_sizes(A, B)
    b = {128: 0, 1024: 1, 8192: 2}[table]
    assert np.all(V.spgemm_bin(ub) == b) and np.all(V.spgemm_bin(nnz) == b) and nnz.max() == table // 2


def test_exact_product_is_exact():
    """the reference against fractions.Fraction on random FP64 rows; cancellation rows give exact zeros in the pattern"""
    A, B = V.spgemm_edges(False, seed=5)
    C, vals, k, asum = V.exact_product(A[:12], B)
    for i in range(3):
        for p in range(C.indptr[i], C.indptr[i + 1]):
            j = C.indices[p]
            terms = [Fraction(float(A.data[q] * B[A.indices[q], j])) for q in range(A.indptr[i], A.indptr[i + 1])
                     if B[A.indices[q], j] != 0]
            assert vals[p] == float(sum(terms)) and k[p] == len(terms)
    A, B = V.spgemm_cancellation()
    C, vals, _, _ = V.exact_product(A, B)
    assert np.count_nonzero(vals == 0.0) == 30 + 200 + 2000 + 5000
    assert np.array_equal(np.diff(C.indptr), [30, 30, 200, 200, 2000, 2000, 5000, 5000])


def test_exact_spmv_matches_fractions():
    A = V.spmv_vector_input(513, 8, seed=3)
    rng = np.random.default_rng(0)
    x, y = rng.standard_normal(A.shape[1]), rng.standard_normal(A.shape[0])
    ref, k, _ = V.exact_spmv(A, x, 2.0, -1.3, y)
    for i in (0, 1, int(np.argmax(np.diff(A.indptr)))):
        lo, hi = A.indptr[i], A.indptr[i + 1]
        s = sum(Fraction(2.0) * Fraction(a) * Fraction(x[j]) for a, j in zip(A.data[lo:hi], A.indices[lo:hi]))
        assert ref[i] == float(s + Fraction(-1.3) * Fraction(y[i])) and k[i] == hi - lo + 2


@pytest.mark.parametrize("tpr", [1, 2, 4, 8, 16, 32])
@pytest.mark.parametrize("longest", [513, 2000, 20000])
def test_spmv_vector_inputs(longest, tpr):
    A = V.spmv_vector_input(longest, tpr, seed=longest + tpr)
    lens = np.diff(A.indptr)
    assert lens.max() == longest and lens.max() > V.STREAM_MAXROW and np.sort(lens)[-2] <= V.STREAM_MAXROW
    assert V.sell_ratio(A) > V.SELL_MAX_RATIO
    assert V.choose_tpr(A.nnz, A.shape[0]) == tpr and V.spmv_path(A) == "VECTOR"
    assert np.any(lens == 0) or tpr >= 16


def test_spmv_threshold_neighbours():
    A = V.spmv_stream_512()
    assert np.diff(A.indptr).max() == 512 and V.sell_ratio(A) > 1.25 and V.spmv_path(A) == "STREAM"
    ratios = {d: V.sell_ratio(V.spmv_sell_padding(d)) for d in (630, 640, 650)}
    assert 1.24 < ratios[630] < 1.25 and ratios[640] == 1.25 and 1.25 < ratios[650] < 1.26
    assert [V.spmv_path(V.spmv_sell_padding(d)) for d in (630, 640, 650)] == ["SELL", "SELL", "STREAM"]


def test_spmv_edge_inputs():
    E = V.spmv_edge_inputs()
    assert E["ragged_1003"].shape[0] % 32 != 0 and np.any(np.diff(E["ragged_1003"].indptr) == 0)
    assert E["single_row_short"].shape[0] == 1 and E["single_row_long"].shape[0] == 1
    assert E["wide_5x100000"].shape[1] > 10000 * E["wide_5x100000"].shape[0]
    assert {k: V.spmv_path(m) for k, m in E.items()} == {"ragged_1003": "STREAM", "single_row_short": "STREAM",
                                                        "single_row_long": "VECTOR", "wide_5x100000": "VECTOR",
                                                        "all_empty_rows": "VECTOR"}


def test_relax_inputs_select_their_tpr_and_are_spd():
    for tpr, A in V.relax_inputs().items():
        assert V.choose_tpr(A.nnz, A.shape[0]) == tpr
        assert abs(A - A.T).max() == 0
        d = A.diagonal()
        assert np.all(d >= np.asarray(abs(A).sum(axis=1)).ravel() - d) and np.all(d > 0)     # diagonally dominant
    assert [V.choose_tpr(n, 1) for n in (0, 1.5, 1.51, 3, 3.1, 6, 6.1, 12, 12.1, 24, 24.1, 100)] == \
        [1, 1, 2, 2, 4, 4, 8, 8, 16, 16, 32, 32]
    assert math.isinf(V.sell_ratio(V._csr([0, 0], [], [], (1, 3))))
