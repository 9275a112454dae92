"""BASELINE configs[4] geometry (examples/3DHdivWeakScaling.cpp: trilinear hexahedra after y += exp(z)/2,
x += sin(y)) through the product path: Coarsen() on the GPU against the oracle, and the reference's own golden
(examples/CMakeLists.txt:130-136) recomputed from the PRODUCT's operators."""
import json
import os

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spl

from parelag_b200 import api, capi
from oracle import amge
from tests.test_coarsen_gpu import compare_levels

pytestmark = pytest.mark.gpu
REF = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_upscaling_norms.json")))


def test_deformed_mesh_coarsen_matches_oracle_and_reference_golden():
    api.session()
    dims, nlev = (4, 4, 4), 3
    mesh, seqs = amge.build_hierarchy(dims, nlev, jstart=2, deform=amge.weak_scaling_deformation)
    S = api.Sequence.hex(dims, nlev, jstart=2, coords=mesh.vertex_coords())
    # (1) sign- and basis-invariant check first: the reference's experiment with the product's P, D and mass operators
    ess = np.array([0, 1, 1, 1, 1, 0])
    i, j = np.meshgrid(np.arange(dims[0]), np.arange(dims[1]), indexing="ij")
    rhs = np.zeros(S.get_csr(0, "M", 2).shape[0])
    rhs[mesh.fz(i.ravel(), j.ravel(), 0)] = 1.0
    sols, Ps = [], [S.get_csr(l, "P", 2) for l in range(nlev - 1)]
    for l in range(nlev):
        M, W, D = S.get_csr(l, "M", 2), S.get_csr(l, "M", 3), S.get_csr(l, "D", 2)
        marker = seqs[l].dof[2].mark_bdr_dofs(ess)
        assert np.array_equal(marker, (S.get_bdr_mask(l, 2) & 0b011110) != 0)
        keep = sp.diags((~marker).astype(float))
        A = keep @ (M + D.T @ W @ D) @ keep + sp.diags(marker.astype(float))
        r = rhs.copy()
        r[marker] = 0.0
        sols.append(spl.spsolve(sp.csc_matrix(A), r))
        if l + 1 < nlev:
            rhs = Ps[l].T @ rhs
    M0, W0, D0 = S.get_csr(0, "M", 2), S.get_csr(0, "M", 3), S.get_csr(0, "D", 2)
    u_err, du_err = [], []
    for l in range(nlev - 1, 0, -1):
        u = sols[l]
        for q in range(l - 1, -1, -1):
            u = Ps[q] @ u
        d = u - sols[0]
        dd = D0 @ d
        u_err.append("%.4e" % np.sqrt(d @ (M0 @ d)))
        du_err.append("%.4e" % np.sqrt(dd @ (W0 @ dd)))
    assert u_err == REF["3DHdivWeakScaling"]["u_errors"] and du_err == REF["3DHdivWeakScaling"]["du_errors"], (u_err, du_err)
    # (2) entry-wise comparison with the oracle (identical SVD sign choices: tie-robust rule, oracle fix_sign / warp_sign_pivot)
    # 58 + 12 NullSpace dofs on this mesh; the level-1 interior ones come from a residual with sigma_2 |T| = 1.6e-4
    # (oracle: singular values 1, 1.5e-2, 2e-12 of a residual of norm 1.1e-2): determined to ~1e-16 / 1.6e-4 * cond
    compare_levels(S, seqs, tol=1e-10, null_tol=1e-8)
    S.free()


def test_deformed_mesh_hcurl_levels_take_the_dense_weighted_trace_svd():
    """Three levels with forms 1-3 on the deformed mesh and variable coefficients: on level 1 the agglomerated edges
    and facets carry several dofs per member entity, their trace mass block is no longer diagonal, and
    ComputeCoarseTraces takes SVD_Calculator::ComputeON(DenseMatrix&W, ...) (ParELAG_SVDCalculator.cpp:258-284:
    SymEigensolver::ComputeAll, X = W^{1/2}) -- in the product a Jacobi eigensolver inside k_traces.  The large local
    problems of level 1 also take the global-workspace variant of the extension kernel."""
    api.session()
    dims, nlev = (4, 4, 4), 3
    rng = np.random.default_rng(11)
    alpha, beta = rng.uniform(0.5, 2.0, 64), 10.0 ** rng.uniform(-1, 1, 64)
    dense = {"n": 0}
    orig = amge.svd_on_weighted

    def spy(M, A):
        dense["n"] += int(np.any(M - np.diag(np.diag(M))))
        return orig(M, A)
    amge.svd_on_weighted = spy
    try:
        mesh, seqs = amge.build_hierarchy(dims, nlev, jstart=1, alpha=alpha, beta=beta, deform=amge.weak_scaling_deformation)
    finally:
        amge.svd_on_weighted = orig
    assert dense["n"] > 0                                       # the oracle really takes the dense-weighted path
    capi.variant_counts(reset=True)
    S = api.Sequence.hex(dims, nlev, jstart=1, alpha=alpha, beta=beta, coords=mesh.vertex_coords())
    assert capi.variant_counts()[capi.EXT_GMEM] > 0
    assert S.stat(2, "trace_dense_mass_1") + S.stat(2, "trace_dense_mass_2") == dense["n"]
    compare_levels(S, seqs, tol=1e-10, null_tol=1e-7)
    # CheckInvariants on the product's own operators (DeRhamSequence.cpp:694-970)
    for l in range(nlev - 1):
        for j in (1, 2, 3):
            P = S.get_csr(l, "P", j)
            Mf, Mc = S.get_csr(l, "M", j), S.get_csr(l + 1, "M", j)
            assert abs(Mc - P.T @ Mf @ P).max() <= 1e-11 * abs(Mc).max(), ("M_c = P^T M P", l, j)
            if j < 3:
                Df, Dc, Pn = S.get_csr(l, "D", j), S.get_csr(l + 1, "D", j), S.get_csr(l, "P", j + 1)
                assert abs(Df @ P - Pn @ Dc).max() <= 1e-11 * max(abs(Df @ P).max(), 1.0), ("D P = P D", l, j)
    S.free()
