"""Oracle-side restatement of the example drivers' algebra (TEST INFRASTRUCTURE ONLY):
system assembly as in examples/MultigridTest{0,1,2}Form.cpp:443-475 and the nested
solver "PCG o AMGe(Hiptmair or l1-GS smoothers, PCG-GS coarse solver)" that the
ParameterList library of examples/testing_helpers/Create{0,1,2}FormParameterList.hpp
describes (coarse solver replaced by the hot-path-only "PCG-GS" of
examples/example_parameterlists/spe10_example_parameters.xml:147-162, SURVEY fact 9)."""
import numpy as np
import scipy.sparse as sp

from . import solve as orc


def system_matrix(seq, form, ess_attr):
    """A = M_form + D^T M_{form+1} D (form 0: D^T M_1 D), essential rows/cols
    eliminated with unit diagonal (SparseMatrix::EliminateRowCol, DIAG_ONE)."""
    D = seq.D[form]
    W = seq.mass_operator(form + 1)
    A = (D.T @ W @ D)
    if form > 0:
        A = A + seq.mass_operator(form)
    A = sp.csr_matrix(A)
    marker = seq.dof[form].mark_bdr_dofs(ess_attr)
    keep = sp.diags((~marker).astype(float))
    A = sp.csr_matrix(keep @ A @ keep + sp.diags(marker.astype(float)))
    A.sum_duplicates(); A.sort_indices()
    return A, marker


def bdr_mask(dofhandler):
    """bit a set <=> dof lies on a facet with boundary attribute a+1"""
    mask = np.zeros(dofhandler.ndofs, dtype=np.uint32)
    fb = dofhandler.topo.facet_bdr
    if dofhandler.mcb < 1:
        return mask
    FD = dofhandler.entity_dof[1]
    for f in range(fb.shape[0]):
        a = fb.indices[fb.indptr[f]:fb.indptr[f + 1]]
        if len(a) == 1:
            mask[FD.indices[FD.indptr[f]:FD.indptr[f + 1]]] |= np.uint32(1 << int(a[0]))
    return mask


# "Type" of the Hypre smoother factory -> hypre relaxation type (ParELAG_HypreSmootherFactory.cpp:27-31)
SMOOTHER_TYPES = {"Jacobi": 0, "L1 Jacobi": 1, "L1 Gauss-Seidel": 2, "L1 Gauss-Seidel Truncated": 4, "Lumped Jacobi": 5,
                  "Gauss-Seidel": 6, "Chebyshev": 16, "Hypre Jacobi": 413}


def gs_order(A, ordering):
    return None if ordering == "natural" else orc.multicolor_order(A)[0]


def amge_pcg_solver(seqs, form, ess_attr, A, ordering="natural", smoother_type=2,
                    coarse_its=3, coarse_tol=1e-4, hiptmair=None, damping=1.0, omega=1.0, cheby_order=2):
    """Returns (prec, info): prec(r) = one AMGe V-cycle.  hiptmair defaults to form>0.  smoother_type: a hypre
    relaxation type or a name of SMOOTHER_TYPES; damping, omega and cheby_order as "Damping Factor", "Omega" and
    "Cheby Poly Order" of library_entries."""
    hiptmair = (form > 0) if hiptmair is None else hiptmair
    stype = SMOOTHER_TYPES[smoother_type] if isinstance(smoother_type, str) else smoother_type
    nl = len(seqs)
    Ps = [seqs[l].get_P(form, ess_attr) for l in range(nl - 1)]

    def kw(M):
        return dict(type=stype, damping=damping, omega=omega, cheby_order=cheby_order,
                    order=gs_order(M, ordering) if stype in (2, 4, 6) else None)

    def hypre(Al):
        return orc.Smoother(Al, **kw(Al))

    def make_smoother(l, Al):
        if not hiptmair:
            return hypre(Al)
        Dl = seqs[l].get_D(form - 1, ess_attr)
        return orc.Hiptmair(Al, Dl, kw, kw)

    def make_coarse(Ac):
        S = make_smoother(nl - 1, Ac)

        def solve(b, x):
            return orc.pcg(Ac, lambda r: S.apply(r, np.zeros_like(r), False), b, rtol=coarse_tol,
                           atol=coarse_tol, max_iter=coarse_its)[0]
        return solve
    H = orc.build_hierarchy(A, Ps, make_smoother, make_coarse)
    return H


def library_entries(form, ordering="natural", smoother="L1 Gauss-Seidel", coarse_its=3, coarse_tol=1e-4,
                    rtol=1e-6, atol=1e-6, max_iter=300, damping=1.0, omega=1.0, cheby_order=2, hiptmair=None):
    """The same solver as a ParElag 'Preconditioner Library' (dict for api.library_xml).  hiptmair defaults to form>0."""
    hiptmair = (form > 0) if hiptmair is None else hiptmair
    hyp = ("Hypre", {"Type": smoother, "Sweeps": 1, "Damping Factor": float(damping), "Omega": float(omega),
                     "Cheby Poly Order": int(cheby_order), "Cheby Poly Fraction": 0.3, "GS ordering": ordering})
    lib = {"Gauss-Seidel": hyp}
    if hiptmair:
        lib["Hiptmair-GS-GS"] = ("Hiptmair", {"Primary Smoother": "Gauss-Seidel", "Auxiliary Smoother": "Gauss-Seidel"})
        smoo = "Hiptmair-GS-GS"
    else:
        smoo = "Gauss-Seidel"
    lib["PCG-GS"] = ("Krylov", {"Solver name": "PCG", "Preconditioner": smoo, "Print level": -1,
                                "Maximum iterations": coarse_its, "Relative tolerance": coarse_tol,
                                "Absolute tolerance": coarse_tol})
    lib["AMGe"] = ("AMGe", {"Maximum levels": -1, "Forms": [form], "PreSmoother": smoo, "PostSmoother": smoo,
                            "Coarse solver": "PCG-GS", "Cycle type": "V-cycle"})
    lib["PCG-AMGe"] = ("Krylov", {"Solver name": "PCG", "Preconditioner": "AMGe", "Print level": -1,
                                  "Maximum iterations": max_iter, "Relative tolerance": rtol,
                                  "Absolute tolerance": atol})
    return lib


# ----------------------------------------------------------------------------
# mixed Darcy system (configs[1] "MultigridTestDarcy", configs[3] SPE10-shaped)
# ----------------------------------------------------------------------------
def darcy_blocks(seq):
    """[[M B^T][B 0]] with M = mass(H(div)), B = W D_2, W = mass(L2) (examples/MultigridTestDarcy.cpp)."""
    M = sp.csr_matrix(seq.mass_operator(2))
    B = orc.spgemm(sp.csr_matrix(seq.mass_operator(3)), sp.csr_matrix(seq.D[2]))
    return M, B


def darcy_library_entries(block="Block Jacobi", ordering="natural", coarse_its=5, coarse_tol=1e-4, rtol=1e-6, atol=1e-6,
                          max_iter=300, restart=50, amge=True, smoother="L1 Gauss-Seidel", s_type="Diagonal"):
    """Parameter list modelled on examples/example_parameterlists/darcy_example_parameters.xml with the
    hypre black boxes (BoomerAMG) replaced by the hot-path l1-Gauss-Seidel smoother (SURVEY fact 9)."""
    lib = {"Gauss-Seidel": ("Hypre", {"Type": smoother, "Sweeps": 1, "Damping Factor": 1.0, "Omega": 1.0,
                                      "GS ordering": ordering})}
    if block == "Block LDU":
        lib["Blk"] = ("Block LDU", {"Damping Factor": 1.0, "A00_1 Inverse": "Gauss-Seidel", "A00_2 Inverse": "Gauss-Seidel",
                                    "A00_3 Inverse": "Gauss-Seidel", "S Inverse": "Gauss-Seidel", "Alpha": 1.0, "S Type": s_type})
    else:
        lib["Blk"] = (block, {"A00 Inverse": "Gauss-Seidel", "A11 Inverse": "Gauss-Seidel", "Alpha": 1.0, "S Type": s_type})
    lib["GMRES-Blk"] = ("Krylov", {"Solver name": "GMRES", "Preconditioner": "Blk", "Print level": -1, "Maximum iterations": coarse_its,
                                   "Relative tolerance": coarse_tol, "Absolute tolerance": coarse_tol, "Restart size": restart})
    lib["AMGe-Blk"] = ("AMGe", {"Maximum levels": -1, "Forms": [2, 3], "PreSmoother": "Blk", "PostSmoother": "Blk",
                                "Coarse solver": "GMRES-Blk", "Cycle type": "V-cycle"})
    lib["GMRES-AMGe-Blk"] = ("Krylov", {"Solver name": "GMRES", "Preconditioner": "AMGe-Blk" if amge else "Blk", "Print level": -1,
                                        "Maximum iterations": max_iter, "Relative tolerance": rtol, "Absolute tolerance": atol,
                                        "Restart size": restart})
    return lib


def darcy_solver(seqs, block="Block Jacobi", ordering="natural", coarse_its=5, coarse_tol=1e-4, restart=50, amge=True,
                 smoother_type=2, s_type="DIAGONAL"):
    """The same solver on the oracle side: returns (A: BlockOp, prec: r -> z).  s_type "MASS": the second diagonal
    operator is ComputeTrueM(forms.front()) of the level's sequence (SchurComplementFactory.cpp:43-50)."""
    M, B = darcy_blocks(seqs[0])
    A0 = orc.BlockOp([[M, sp.csr_matrix(B.T)], [B, None]])

    def gs(Mx):
        S = orc.Smoother(Mx, type=smoother_type, order=gs_order(Mx, ordering) if smoother_type == 2 else None)
        return lambda r: S.apply(r, np.zeros_like(r), False)

    def make_smoother(l, A):
        A00, A01, A10, A11 = A.blocks[0][0], A.blocks[0][1], A.blocks[1][0], A.blocks[1][1]
        negS = sp.csr_matrix(orc.schur_complement(A00, A01, A10, A11, 1.0, s_type) * (-1.0))
        if block == "Block Jacobi":
            return orc.BlockJacobi(A, [gs(A00), gs(negS)])
        if block == "Block GS":
            return orc.BlockGS(A, [gs(A00), gs(negS)])
        return orc.BlockLDU(A, gs(A00), gs(A00), gs(A00), gs(negS), 1.0)
    if not amge:
        S = make_smoother(0, A0)
        return A0, (lambda r: S.apply(r, np.zeros_like(r), False))

    def make_coarse(Ac):
        S = make_smoother(len(seqs) - 1, Ac)
        return lambda b, x: orc.gmres(Ac.mult, lambda r: S.apply(r, np.zeros_like(r), False), b, rtol=coarse_tol, atol=coarse_tol,
                                      max_iter=coarse_its, restart=restart)[0]
    Ps = [[sp.csr_matrix(seqs[l].get_P(2)), sp.csr_matrix(seqs[l].get_P(3))] for l in range(len(seqs) - 1)]
    H = orc.build_block_hierarchy(A0, Ps, [False, False], make_smoother, make_coarse)
    return A0, H.mult
