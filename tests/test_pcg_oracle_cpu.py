"""The oracle's PCG (mfem::CGSolver::Mult restated) on operators that are not positive definite, in exact arithmetic:
a negative (Ad, d) goes on with a negative step, only an exact zero stops.  The GPU's host and device-resident PCG loops
are compared with it in test_vcycle_modes_gpu.py."""
import numpy as np
import scipy.sparse as sp

from oracle import solve as orc

N = 8


def test_negative_curvature_takes_a_negative_step():
    A = sp.diags(-np.ones(N), format="csr")
    x, it, conv, hist = orc.pcg(A, None, np.ones(N), rtol=1e-6, atol=0.0, max_iter=5)
    assert (it, conv, hist) == (1, True, [N, 0.0])
    assert np.array_equal(x, -np.ones(N))


def test_zero_curvature_stops_unconverged():
    A = sp.diags(np.where(np.arange(N) % 2 == 0, 1.0, 0.0), format="csr")
    # first check: b lies in the null space
    x, it, conv, hist = orc.pcg(A, None, np.where(np.arange(N) % 2 == 1, 1.0, 0.0), rtol=0.0, atol=0.0, max_iter=5)
    assert (it, conv, hist) == (0, False, [N / 2]) and not x.any()
    # in the loop: d_1 = r_1 + d_0 lies in the null space; the count is the iteration that computed (Ad, d)
    x, it, conv, hist = orc.pcg(A, None, np.ones(N), rtol=0.0, atol=0.0, max_iter=5)
    assert (it, conv, hist) == (2, False, [N, N])
    assert np.array_equal(x, 2.0 * np.ones(N))


def test_negative_initial_norm_stops_at_once():
    A = sp.diags(-2.0 * np.ones(N), format="csr")
    x, it, conv, hist = orc.pcg(A, lambda r: r / A.diagonal(), np.ones(N), rtol=1e-6, atol=0.0, max_iter=5)
    assert (it, conv, hist) == (0, False, [-N / 2]) and not x.any()
