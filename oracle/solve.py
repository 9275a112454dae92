"""Oracle (TEST INFRASTRUCTURE ONLY) for ParElag's AMGe *solve* path.

CPU restatement, single threaded and deterministic, of
  * the V-cycle        src/linalg/solver_ops/ParELAG_Hierarchy.cpp:109-253
  * the hierarchy      src/linalg/solver_ops/ParELAG_Hierarchy.cpp:282-383
  * Hiptmair smoother  src/linalg/solver_ops/ParELAG_HiptmairSmoother.cpp:48-109,
                       src/linalg/factories/ParELAG_HiptmairSmootherFactory.cpp:52-179
  * hypre relaxation   behind src/linalg/solver_ops/ParELAG_HypreSmootherWrapper.cpp:20-35
  * PCG                mfem::CGSolver::Mult behind src/linalg/solver_ops/ParELAG_KrylovSolver.cpp:23-96
The arithmetic kernels are the plain-C functions of oracle/solve_oracle.c (hypre /
MFEM algorithms restated from their published form -- those libraries are not
vendored in the reference tree; "parity unpinned" at kernel level, SURVEY.md 8c).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
may import this module.  The product (parelag_b200/) never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import scipy.sparse as sp

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libsolve_oracle.so")
_lib = None


def build():
    src = os.path.join(_HERE, "solve_oracle.c")
    if (not os.path.exists(_SO)) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-fopenmp", "-fPIC", "-shared",
                               "-o", _SO, src, "-lm"])


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _csr(A):
    A = A.tocsr()
    return (A.shape[0], np.ascontiguousarray(A.indptr, dtype=np.int32),
            np.ascontiguousarray(A.indices, dtype=np.int32),
            np.ascontiguousarray(A.data, dtype=np.float64))


_THREADS = 1
_T_CACHE = {}


def set_threads(n):
    """CPU-baseline timing legs only: n OpenMP threads for SpMV (rows are independent: same result) and for the
    blocked hybrid Gauss-Seidel; A^T x goes through a cached explicit transpose (what hypre's MatvecT costs per
    rank).  Returns the number of threads a parallel region really gets."""
    global _THREADS
    lib().orc_set_num_threads(int(n))
    _THREADS = int(n)
    _T_CACHE.clear()
    return int(lib().orc_probe_threads())


def matvec(A, x, alpha=1.0, beta=0.0, y=None, threads=False):
    threads = threads or _THREADS > 1
    n, I, J, D = _csr(A)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.zeros(n) if y is None else np.ascontiguousarray(y, dtype=np.float64).copy()
    f = lib().orc_csr_matvec_mt if threads else lib().orc_csr_matvec
    f(n, _p(I), _p(J), _p(D), C.c_double(alpha), _p(x), C.c_double(beta), _p(y))
    return y


def matvec_t(A, x, alpha=1.0, beta=0.0, y=None):
    if _THREADS > 1:
        key = id(A)
        if key not in _T_CACHE:
            _T_CACHE[key] = (A, sp.csr_matrix(A.T))       # keep A alive: id() stays unique
        return matvec(_T_CACHE[key][1], x, alpha=alpha, beta=beta, y=y, threads=True)
    n, I, J, D = _csr(A)
    m = A.shape[1]
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.zeros(m) if y is None else np.ascontiguousarray(y, dtype=np.float64).copy()
    lib().orc_csr_matvec_t(n, m, _p(I), _p(J), _p(D), C.c_double(alpha), _p(x), C.c_double(beta), _p(y))
    return y


def l1_norms(A, option):
    n, I, J, D = _csr(A)
    l1 = np.empty(n)
    lib().orc_l1_norms(n, _p(I), _p(J), _p(D), None, None, option, _p(l1))
    return l1


def greedy_colors(A):
    """First-fit colouring, rows visited in natural order, smallest colour not used
    by an already-coloured neighbour in the row pattern (spec shared with the GPU)."""
    n, I, J, _ = _csr(A)
    color = np.empty(n, dtype=np.int32)
    ncol = lib().orc_greedy_colors(n, _p(I), _p(J), _p(color))
    return color, ncol


def multicolor_order(A):
    color, ncol = greedy_colors(A)
    return np.argsort(color, kind="stable").astype(np.int32), ncol


def natural_levels(A):
    """level(i) = 1 + max level(j), j<i coupled: the DAG schedule that reproduces a
    sequential natural-order sweep."""
    n, I, J, _ = _csr(A)
    level = np.zeros(n, dtype=np.int32)
    for i in range(n):
        l = 0
        for j in J[I[i]:I[i + 1]]:
            if j < i and level[j] + 1 > l:
                l = level[j] + 1
        level[i] = l
    return level


def fix_zero_rows(A):
    n, I, J, D = _csr(A)
    D = D.copy()
    nf = lib().orc_fix_zero_rows(n, _p(I), _p(J), _p(D), None, None)
    return sp.csr_matrix((D, J, I), shape=A.shape), nf


def spgemm(A, B):
    """C = A*B with sorted columns, explicit zeros kept."""
    n, AI, AJ, AA = _csr(A)
    _, BI, BJ, BA = _csr(B)
    CI = np.zeros(n + 1, dtype=np.int32)
    nnz = lib().orc_spgemm_symbolic(n, _p(AI), _p(AJ), _p(BI), _p(BJ), B.shape[1], _p(CI))
    CJ = np.zeros(max(nnz, 1), dtype=np.int32)
    CA = np.zeros(max(nnz, 1))
    lib().orc_spgemm_numeric(n, _p(AI), _p(AJ), _p(AA), _p(BI), _p(BJ), _p(BA), B.shape[1],
                             _p(CI), _p(CJ), _p(CA))
    return _raw_csr(CA[:nnz], CJ[:nnz], CI, (n, B.shape[1]))


def _raw_csr(data, indices, indptr, shape):
    # build without scipy's canonicalisation so explicit zeros / order survive
    M = sp.csr_matrix(shape)
    M.data, M.indices, M.indptr = data, indices, indptr
    return M


def transpose(A):
    n, I, J, D = _csr(A)
    m = A.shape[1]
    TI = np.zeros(m + 1, dtype=np.int32)
    TJ = np.zeros(max(len(J), 1), dtype=np.int32)
    TA = np.zeros(max(len(J), 1))
    lib().orc_csr_transpose(n, m, _p(I), _p(J), _p(D), _p(TI), _p(TJ), _p(TA))
    return _raw_csr(TA[:len(J)], TJ[:len(J)], TI, (m, n))


def rap(A, P, R=None):
    """R^T A P (R = P when None): mfem::RAP, Hierarchy.cpp:365."""
    Rt = transpose(P if R is None else R)
    return spgemm(Rt, spgemm(A, P))


def hypre_rand_vector(n, seed=1):
    v = np.empty(n)
    lib().orc_hypre_rand_vector(n, seed, _p(v))
    return v


class Smoother:
    """mfem::HypreSmoother as configured by parelag::HypreSmootherWrapper.  type 413 ("Hypre Jacobi") is
    mfem::HypreDiagScale: x = diag(A)^{-1} b, one unit-weight Jacobi sweep from a zero guess whatever the
    initial guess, sweeps and damping."""

    def __init__(self, A, type=2, sweeps=1, damping=1.0, omega=1.0, cheby_order=2,
                 cheby_fraction=0.3, order=None, ranks=1):
        """ranks > 1 (CPU-baseline timing only, type 2): the matrix rows are split into
        `ranks` contiguous blocks handled by one thread each -- Gauss-Seidel inside a block,
        Jacobi across blocks, l1 norms with the off-block part: what the reference computes
        on `ranks` MPI ranks."""
        self.ranks = ranks
        self.A = A.tocsr()
        self.n, self.I, self.J, self.D = _csr(self.A)
        self.type, self.sweeps, self.w, self.omega = type, sweeps, damping, omega
        if type == 413:
            self.sweeps, self.w = 1, 1.0
        l1opt = 0 if type in (0, 6, 16, 413) else type
        self.l1 = l1_norms(self.A, l1opt)
        if ranks > 1:
            assert type == 2 and order is None
            lib().orc_l1_norms_blocked(self.n, _p(self.I), _p(self.J), _p(self.D), ranks, _p(self.l1))
        self.order = None if order is None else np.ascontiguousarray(order, dtype=np.int32)
        self.rank_of_row = None
        if self.order is not None:
            self.rank_of_row = np.empty(self.n, dtype=np.int32)
            self.rank_of_row[self.order] = np.arange(self.n, dtype=np.int32)
        if type == 16:
            self.max_eig, self.min_eig = self._eig_estimate_cg(10)
            self.coefs = np.zeros(5)
            self.cheby_order = lib().orc_cheby_coefs(C.c_double(self.max_eig), C.c_double(self.min_eig),
                                                     C.c_double(cheby_fraction), cheby_order, _p(self.coefs))

    def _eig_estimate_cg(self, max_iter):
        """hypre_ParCSRMaxEigEstimateCG(A, scale=1, max_iter)."""
        n = self.n
        max_iter = min(max_iter, n)
        ds = 1.0 / np.sqrt(self.A.diagonal())
        r = hypre_rand_vector(n, 1)
        tridiag = np.zeros(max_iter + 1)
        trioffd = np.zeros(max_iter + 1)
        gamma = float(r @ r)
        p = None
        for i in range(max_iter):
            s = r.copy()
            gamma_old = gamma
            gamma = float(r @ s)
            if i > 0 and gamma < 2.220446049250313e-16:     # residual gone: the Lanczos matrix so far
                max_iter = i
                break
            if i == 0:
                beta = 1.0
                p = s.copy()
            else:
                beta = gamma / gamma_old
                p = s + beta * p
            s = ds * matvec(self.A, ds * p)
            sdotp = float(s @ p)
            alpha = gamma / sdotp
            alphainv = 1.0 / alpha
            tridiag[i + 1] = alphainv
            tridiag[i] *= beta
            tridiag[i] += alphainv
            trioffd[i + 1] = alphainv
            trioffd[i] *= np.sqrt(beta)
            r = r - alpha * s
        T = np.diag(tridiag[:max_iter]) + np.diag(trioffd[1:max_iter], 1) + np.diag(trioffd[1:max_iter], -1)
        ev = np.linalg.eigvalsh(T)
        return float(ev[-1]), float(ev[0])

    def apply(self, b, x, iterative_mode=True):
        b = np.ascontiguousarray(b, dtype=np.float64)
        x = np.ascontiguousarray(x, dtype=np.float64).copy()
        if not iterative_mode or self.type == 413:
            x[:] = 0.0
        n = self.n
        for _ in range(self.sweeps):
            if self.type in (0, 1, 5, 413):
                v = np.empty(n)
                lib().orc_relax_jacobi(n, _p(self.I), _p(self.J), _p(self.D), None, None, None,
                                       _p(self.l1), C.c_double(self.w), _p(b), _p(x), None, _p(v))
            elif self.type == 2 and self.ranks > 1:
                frozen = np.empty(n)
                lib().orc_relax_gs_blocked(n, _p(self.I), _p(self.J), _p(self.D), _p(self.l1), self.ranks,
                                           _p(b), _p(x), _p(frozen))
            elif self.type in (2, 4, 6):
                uold = np.empty(n)
                lib().orc_relax_gs(n, _p(self.I), _p(self.J), _p(self.D), None, None, None,
                                   _p(self.l1), C.c_double(self.w), C.c_double(self.omega),
                                   _p(self.order), _p(self.rank_of_row), _p(b), _p(x), None, _p(uold))
            elif self.type == 16:
                work = np.empty(5 * n)
                lib().orc_relax_cheby(n, _p(self.I), _p(self.J), _p(self.D), _p(self.coefs),
                                      self.cheby_order, _p(b), _p(x), _p(work))
            else:
                raise ValueError("unsupported smoother type %d" % self.type)
        return x


class Hiptmair:
    """parelag::HiptmairSmoother (HiptmairSmoother.cpp:48-76): primary smooth, residual,
    D^T r, auxiliary smooth from zero, x += D x_aux.  A_aux = D^T A D + FixZeroRows
    (HiptmairSmootherFactory.cpp:143-165)."""

    def __init__(self, A, D, primary_kw, aux_kw):
        self.A, self.Dm = A.tocsr(), D.tocsr()
        Aaux, _ = fix_zero_rows(rap(self.A, self.Dm))
        self.A_aux = Aaux
        self.primary = Smoother(self.A, **primary_kw(self.A))
        self.aux = Smoother(self.A_aux, **aux_kw(self.A_aux))

    def apply(self, b, x, iterative_mode=True):
        if not iterative_mode:
            x = np.zeros_like(x)
        x = self.primary.apply(b, x, True)
        r = matvec(self.A, x, alpha=-1.0, beta=1.0, y=b)
        auxb = matvec_t(self.Dm, r)
        auxx = self.aux.apply(auxb, np.zeros(self.Dm.shape[1]), False)
        return x + matvec(self.Dm, auxx)


    def apply_transpose(self, b, x, iterative_mode=True):
        """HiptmairSmoother::MultTranspose (HiptmairSmoother.cpp:79-109): auxiliary correction first (from B itself in
        preconditioner mode, from the residual otherwise), then the primary sweep."""
        if not iterative_mode:
            x = np.zeros_like(x)
            auxb = matvec_t(self.Dm, b)
        else:
            auxb = matvec_t(self.Dm, matvec(self.A, x, alpha=-1.0, beta=1.0, y=b))
        auxx = self.aux.apply(auxb, np.zeros(self.Dm.shape[1]), False)
        x = x + matvec(self.Dm, auxx)
        return self.primary.apply(b, x, True)


def stationary(A, corrector, b, rtol=0.0, atol=0.0, max_iter=1, x0=None):
    """StationarySolver::Mult (ParELAG_StationarySolver.cpp:41-147): x += S r, r -= A (S r) (the residual is updated,
    not recomputed); stops on ||r|| < atol, accumulated ratio < rtol, a zero correction, or max_iter.
    corrector(r) -> S r from a zero initial guess.  Returns (x, iterations, converged, [||r_k||])."""
    b = np.asarray(b, dtype=np.float64)
    if x0 is None:
        x, r = np.zeros_like(b), b.copy()
    else:
        x = np.array(x0, dtype=np.float64)
        r = -matvec(A, x) + b
    nk1 = float(np.sqrt(r @ r))
    hist, its, ratio, conv = [nk1], 0, 1.0, False
    while its < max_iter:
        its += 1
        c = corrector(r)
        x = x + c
        r = r - matvec(A, c)
        nk = float(np.sqrt(r @ r))
        hist.append(nk)
        ratio *= nk / nk1
        if nk < atol or ratio < rtol:
            conv = True
            break
        if nk / nk1 == 1.0:
            break
        nk1 = nk
    return x, its, conv, hist


class Hierarchy:
    """parelag::Hierarchy: levels[l] = dict(A=, P= (to level l from l+1, stored on l+1
    in the reference; here stored on the finer level l as 'P'), pre=, post=), coarsest
    level has 'coarse'.  Mult == one V-cycle from a zero initial guess (Hierarchy.cpp:109-136)."""

    def __init__(self, levels):
        self.levels = levels

    def iterate(self, rhs, sol, l=0):
        L = self.levels[l]
        if l == len(self.levels) - 1:
            return L["coarse"](rhs, sol)
        if L.get("pre") is not None:
            sol = L["pre"].apply(rhs, sol, True)
        resid = matvec(L["A"], sol, alpha=-1.0, beta=1.0, y=rhs)
        crhs = matvec_t(L["P"], resid)
        csol = self.iterate(crhs, np.zeros(L["P"].shape[1]), l + 1)
        sol = sol + matvec(L["P"], csol)
        if L.get("post") is not None:
            sol = L["post"].apply(rhs, sol, True)
        return sol

    def mult(self, rhs):
        return self.iterate(np.asarray(rhs, dtype=np.float64), np.zeros(len(rhs)), 0)


def pcg(A, prec, b, rtol=1e-6, atol=1e-6, max_iter=300, x0=None):
    """mfem::CGSolver::Mult (iterative_mode=false unless x0 is given).  Returns
    (x, iterations, converged, history) with history[i] = (B r, r) after iteration
    i (history[0] is the initial value) -- the quantity MFEM prints and the parity
    contract compares."""
    Amul = (lambda v: matvec(A, v)) if sp.issparse(A) else A
    b = np.asarray(b, dtype=np.float64)
    if x0 is None:
        x = np.zeros_like(b)
        r = b.copy()
    else:
        x = np.array(x0, dtype=np.float64)
        r = b - Amul(x)
    z = prec(r) if prec is not None else r.copy()
    d = z.copy()
    nom0 = nom = float(d @ r)
    hist = [nom]
    if nom < 0:
        return x, 0, False, hist
    r0 = max(nom * rtol * rtol, atol * atol)
    if nom <= r0:
        return x, 0, True, hist
    z = Amul(d)
    den = float(z @ d)
    # a negative (Ad, d) is only reported by MFEM and the iteration goes on; an exact zero stops it
    if den == 0:
        return x, 0, False, hist
    i = 1
    converged = False
    while True:
        alpha = nom / den
        x = x + alpha * d
        r = r - alpha * z
        z = prec(r) if prec is not None else r.copy()
        betanom = float(r @ z)
        hist.append(betanom)
        if betanom < r0:
            converged = True
            break
        i += 1
        if i > max_iter:
            break
        beta = betanom / nom
        d = z + beta * d
        z = Amul(d)
        den = float(d @ z)
        if den == 0:
            break
        nom = betanom
    return x, min(i, max_iter), converged, hist


def build_hierarchy(A0, Ps, make_smoother, make_coarse):
    """buildHierarchyFromDeRhamSequence (Hierarchy.cpp:282-383): A_{l+1} = P_l^T A_l P_l,
    then FixZeroRows; smoothers per AMGeSolverFactory.cpp:74-166."""
    levels = []
    A = A0.tocsr()
    for l, P in enumerate(Ps):
        levels.append({"A": A, "P": P.tocsr()})
        A, _ = fix_zero_rows(rap(A, P.tocsr()))
    levels.append({"A": A})
    for l, L in enumerate(levels[:-1]):
        L["pre"] = make_smoother(l, L["A"])
        L["post"] = L["pre"]
    levels[-1]["coarse"] = make_coarse(levels[-1]["A"])
    return Hierarchy(levels)


# ----------------------------------------------------------------------------
# mixed (Darcy) path: GMRES, block preconditioners, Schur complement, blocked hierarchy
# ----------------------------------------------------------------------------
def gmres(A, prec, b, rtol=1e-6, atol=1e-6, max_iter=300, restart=50, x0=None):
    """mfem::GMRESSolver::Mult (left preconditioning, modified Gram-Schmidt, Givens rotations; "the
    algorithm on p. 20 of the SIAM Templates book").  MFEM is third-party and not vendored in the
    reference: restated from the published algorithm, parity unpinned.  Returns
    (x, iterations, converged, history) with history[i] = ||B r|| after iteration i."""
    Amul = (lambda v: matvec(A, v)) if sp.issparse(A) else A
    b = np.asarray(b, dtype=np.float64)
    n, m = len(b), restart
    x = np.zeros(n) if x0 is None else np.array(x0, dtype=np.float64)
    if x0 is None:
        r = prec(b) if prec is not None else b.copy()
    else:
        w = b - Amul(x)
        r = prec(w) if prec is not None else w
    beta = float(np.sqrt(r @ r))
    hist = [beta]
    final_norm = max(rtol * beta, atol)
    if beta <= final_norm:
        return x, 0, True, hist

    def gen_rot(dx, dy):
        if dy == 0.0:
            return 1.0, 0.0
        if abs(dy) > abs(dx):
            t = dx / dy
            sn = 1.0 / np.sqrt(1.0 + t * t)
            return t * sn, sn
        t = dy / dx
        cs = 1.0 / np.sqrt(1.0 + t * t)
        return cs, t * cs

    def app_rot(dx, dy, cs, sn):
        return cs * dx + sn * dy, -sn * dx + cs * dy

    def update(x, k, H, s, V):
        y = s[:k + 1].copy()
        for i in range(k, -1, -1):
            y[i] /= H[i, i]
            for j in range(i - 1, -1, -1):
                y[j] -= H[j, i] * y[i]
        for j in range(k + 1):
            x = x + y[j] * V[j]
        return x
    j = 1
    while j <= max_iter:
        H = np.zeros((m + 1, m)); s = np.zeros(m + 1); cs = np.zeros(m + 1); sn = np.zeros(m + 1)
        V = [r / beta]
        s[0] = beta
        i = 0
        while i < m and j <= max_iter:
            w = Amul(V[i])
            if prec is not None:
                w = prec(w)
            for k in range(i + 1):
                H[k, i] = float(w @ V[k])
                w = w - H[k, i] * V[k]
            H[i + 1, i] = float(np.sqrt(w @ w))
            V.append(w / H[i + 1, i])
            for k in range(i):
                H[k, i], H[k + 1, i] = app_rot(H[k, i], H[k + 1, i], cs[k], sn[k])
            cs[i], sn[i] = gen_rot(H[i, i], H[i + 1, i])
            H[i, i], H[i + 1, i] = app_rot(H[i, i], H[i + 1, i], cs[i], sn[i])
            s[i], s[i + 1] = app_rot(s[i], s[i + 1], cs[i], sn[i])
            resid = abs(s[i + 1])
            hist.append(float(resid))
            if resid <= final_norm:
                return update(x, i, H, s, V), j, True, hist
            i += 1; j += 1
        x = update(x, i - 1, H, s, V)
        w = b - Amul(x)
        r = prec(w) if prec is not None else w
        beta = float(np.sqrt(r @ r))
        if beta <= final_norm:
            return x, j, True, hist
    return x, max_iter, False, hist


def schur_complement(A00, A01, A10, A11=None, alpha=1.0, kind="DIAGONAL"):
    """SchurComplementFactory::BuildOperator (SchurComplementFactory.cpp:51-166):
    A11 - alpha A10 diag(A00)^{-1} A01 (DIAGONAL) or with absolute row sums (ABSROWSUM)."""
    d = A00.diagonal() if kind.upper() == "DIAGONAL" else np.asarray(abs(A00).sum(axis=1)).ravel()
    prod = spgemm(A10.tocsr(), sp.csr_matrix(sp.diags(1.0 / d) @ A01.tocsr()))
    if A11 is None:
        return sp.csr_matrix(prod * (-alpha))
    return sp.csr_matrix(A11 - alpha * prod)


class BlockOp:
    """MfemBlockOperator: blocks[i][j] scipy matrices or None; offsets from the block sizes."""

    def __init__(self, blocks):
        self.blocks = [[None if b is None else b.tocsr() for b in row] for row in blocks]
        nb = len(blocks)
        sizes = []
        for i in range(nb):
            h = next((b.shape[0] for b in self.blocks[i] if b is not None), None)
            if h is None:
                h = next(self.blocks[j][i].shape[1] for j in range(nb) if self.blocks[j][i] is not None)
            sizes.append(h)
        self.off = np.concatenate([[0], np.cumsum(sizes)])
        self.shape = (self.off[-1], self.off[-1])

    def blk(self, v, i):
        return v[self.off[i]:self.off[i + 1]]

    def mult(self, x):
        y = np.zeros(self.off[-1])
        for i, row in enumerate(self.blocks):
            for j, b in enumerate(row):
                if b is not None:
                    y[self.off[i]:self.off[i + 1]] += matvec(b, self.blk(x, j))
        return y


class BlockJacobi:
    """BlockDiagonalSolver with the Block2x2JacobiSolverFactory wiring (S = -Schur complement when
    use_negative_s).  inv[i](r) applies the block inverse from a zero guess."""

    def __init__(self, A, inv):
        self.A, self.inv = A, inv

    def apply(self, b, x, iterative_mode=True):
        if not iterative_mode:
            r, base = np.asarray(b, dtype=np.float64), np.zeros_like(b)
        else:
            r, base = b - self.A.mult(x), x
        c = np.zeros_like(r)
        for i, f in enumerate(self.inv):
            c[self.A.off[i]:self.A.off[i + 1]] = f(self.A.blk(r, i))
        return base + c


class BlockGS:
    """BlockTriangularSolver, lower triangle (Block2x2GaussSeidelSolverFactory)."""

    def __init__(self, A, inv):
        self.A, self.inv = A, inv

    def apply(self, b, x, iterative_mode=True):
        if not iterative_mode:
            r, base = np.asarray(b, dtype=np.float64), np.zeros_like(b)
        else:
            r, base = b - self.A.mult(x), x
        c = np.zeros_like(r)
        for i, f in enumerate(self.inv):
            t = self.A.blk(r, i).copy()
            for j in range(i):
                if self.A.blocks[i][j] is not None:
                    t -= matvec(self.A.blocks[i][j], self.A.blk(c, j))
            c[self.A.off[i]:self.A.off[i + 1]] = f(t)
        return base + c


class BlockLDU:
    """Block2x2LDUInverseOperator::Mult (Block2x2LDUInverseOperator.cpp:73-135)."""

    def __init__(self, A, inv1, inv2, inv3, invS, damping=1.0):
        self.A, self.inv1, self.inv2, self.inv3, self.invS, self.damping = A, inv1, inv2, inv3, invS, damping

    def apply(self, b, x, iterative_mode=True):
        A = self.A
        r = np.asarray(b, dtype=np.float64).copy() if not iterative_mode else b - A.mult(x)
        r0, r1 = A.blk(r, 0), A.blk(r, 1).copy()
        t0 = self.inv2(r0)
        r1 -= matvec(A.blocks[1][0], t0)
        dp = self.invS(r1)
        t = self.inv3(matvec(A.blocks[0][1], dp))
        du = self.inv1(r0) - t
        c = self.damping * np.concatenate([du, dp])
        return c if not iterative_mode else x + c


def build_block_hierarchy(A0, P_blocks_per_level, ess_flags, make_smoother, make_coarse):
    """buildBlockedHierarchyFromDeRhamSequence (Hierarchy.cpp:400-544): A_c(i,j) = P_i^T A(i,j) P_j,
    FixZeroRows on diagonal blocks that carry essential conditions; P = blockdiag(P_i)."""
    levels = []
    A = A0
    for Pb in P_blocks_per_level:
        nb = len(Pb)
        Ac = [[None] * nb for _ in range(nb)]
        for i in range(nb):
            for j in range(nb):
                if A.blocks[i][j] is not None:
                    t = rap(A.blocks[i][j], Pb[j].tocsr(), R=Pb[i].tocsr())
                    if i == j and ess_flags[i]:
                        t, _ = fix_zero_rows(t)
                    Ac[i][j] = t
        levels.append({"A": A, "P": sp.block_diag([p.tocsr() for p in Pb], format="csr")})
        A = BlockOp(Ac)
    levels.append({"A": A})
    for l, L in enumerate(levels[:-1]):
        L["pre"] = make_smoother(l, L["A"])
        L["post"] = L["pre"]
    levels[-1]["coarse"] = make_coarse(levels[-1]["A"])
    return BlockHierarchy(levels)


class BlockHierarchy(Hierarchy):
    def iterate(self, rhs, sol, l=0):
        L = self.levels[l]
        if l == len(self.levels) - 1:
            return L["coarse"](rhs, sol)
        if L.get("pre") is not None:
            sol = L["pre"].apply(rhs, sol, True)
        resid = rhs - L["A"].mult(sol)
        crhs = matvec_t(L["P"], resid)
        csol = self.iterate(crhs, np.zeros(L["P"].shape[1]), l + 1)
        sol = sol + matvec(L["P"], csol)
        if L.get("post") is not None:
            sol = L["post"].apply(rhs, sol, True)
        return sol


def fgmres(A, prec, b, rtol=1e-6, atol=1e-6, max_iter=300, restart=50):
    """mfem::FGMRESSolver::Mult (flexible, right-preconditioned; history = || r ||); restated, parity unpinned."""
    Amul = (lambda v: matvec(A, v)) if sp.issparse(A) else A
    b = np.asarray(b, dtype=np.float64)
    n, m = len(b), restart
    x, r = np.zeros(n), b.copy()
    beta = float(np.sqrt(r @ r))
    hist = [beta]
    final_norm = max(rtol * beta, atol)
    if beta <= final_norm:
        return x, 0, True, hist

    def gen_rot(dx, dy):
        if dy == 0.0:
            return 1.0, 0.0
        if abs(dy) > abs(dx):
            t = dx / dy
            sn = 1.0 / np.sqrt(1.0 + t * t)
            return t * sn, sn
        t = dy / dx
        cs = 1.0 / np.sqrt(1.0 + t * t)
        return cs, t * cs
    rot = lambda dx, dy, c, s: (c * dx + s * dy, -s * dx + c * dy)

    def update(x, k, H, s, Z):
        y = s[:k + 1].copy()
        for i in range(k, -1, -1):
            y[i] /= H[i, i]
            for j in range(i - 1, -1, -1):
                y[j] -= H[j, i] * y[i]
        for j in range(k + 1):
            x = x + y[j] * Z[j]
        return x
    j = 1
    while j <= max_iter:
        H = np.zeros((m + 1, m)); s = np.zeros(m + 1); cs = np.zeros(m + 1); sn = np.zeros(m + 1)
        V, Z = [r / beta], []
        s[0] = beta
        i = 0
        while i < m and j <= max_iter:
            Z.append(prec(V[i]) if prec is not None else V[i].copy())
            r = Amul(Z[i])
            for k in range(i + 1):
                H[k, i] = float(r @ V[k])
                r = r - H[k, i] * V[k]
            H[i + 1, i] = float(np.sqrt(r @ r))
            V.append(r / H[i + 1, i])
            for k in range(i):
                H[k, i], H[k + 1, i] = rot(H[k, i], H[k + 1, i], cs[k], sn[k])
            cs[i], sn[i] = gen_rot(H[i, i], H[i + 1, i])
            H[i, i], H[i + 1, i] = rot(H[i, i], H[i + 1, i], cs[i], sn[i])
            s[i], s[i + 1] = rot(s[i], s[i + 1], cs[i], sn[i])
            resid = abs(s[i + 1])
            hist.append(float(resid))
            if resid <= final_norm:
                return update(x, i, H, s, Z), j, True, hist
            i += 1; j += 1
        x = update(x, i - 1, H, s, Z)
        r = b - Amul(x)
        beta = float(np.sqrt(r @ r))
        if beta <= final_norm:
            return x, j, True, hist
    return x, max_iter, False, hist


def bicgstab(A, prec, b, rtol=1e-6, atol=1e-6, max_iter=300):
    """mfem::BiCGSTABSolver::Mult; history[i] = ||r|| after iteration i; restated, parity unpinned."""
    Amul = (lambda v: matvec(A, v)) if sp.issparse(A) else A
    M = prec if prec is not None else (lambda v: v.copy())
    b = np.asarray(b, dtype=np.float64)
    x, r = np.zeros_like(b), b.copy()
    rt = r.copy()
    resid = float(np.sqrt(r @ r))
    hist = [resid]
    goal = max(resid * rtol, atol)
    if resid <= goal:
        return x, 0, True, hist
    rho_2 = alpha = omega = 1.0
    p = v = None
    for i in range(1, max_iter + 1):
        rho_1 = float(rt @ r)
        if rho_1 == 0.0:
            return x, i, False, hist
        if i == 1:
            p = r.copy()
        else:
            beta = (rho_1 / rho_2) * (alpha / omega)
            p = p - omega * v
            p = r + beta * p
        phat = M(p)
        v = Amul(phat)
        alpha = rho_1 / float(rt @ v)
        s = r - alpha * v
        resid = float(np.sqrt(s @ s))
        if resid < goal:
            hist.append(resid)
            return x + alpha * phat, i, True, hist
        shat = M(s)
        t = Amul(shat)
        omega = float(t @ s) / float(t @ t)
        x = x + alpha * phat
        x = x + omega * shat
        r = s - omega * t
        rho_2 = rho_1
        resid = float(np.sqrt(r @ r))
        hist.append(resid)
        if resid < goal:
            return x, i, True, hist
        if omega == 0.0:
            return x, i, False, hist
    return x, max_iter, False, hist


def minres(A, prec, b, rtol=1e-6, atol=1e-6, max_iter=300):
    """mfem::MINRESSolver::Mult (van der Vorst Fig. 6.9 with an SPD preconditioner); history = |eta|;
    restated, parity unpinned."""
    Amul = (lambda v: matvec(A, v)) if sp.issparse(A) else A
    b = np.asarray(b, dtype=np.float64)
    x = np.zeros_like(b)
    v1 = b.copy()
    u1 = prec(v1) if prec is not None else None
    z = u1 if prec is not None else v1
    eta = beta = float(np.sqrt(z @ v1))
    hist = [eta]
    goal = max(rtol * eta, atol)
    gamma0 = gamma1 = 1.0
    sigma0 = sigma1 = 0.0
    v0 = np.zeros_like(b); w0 = np.zeros_like(b); w1 = np.zeros_like(b)
    if eta <= goal:
        return x, 0, True, hist
    for it in range(1, max_iter + 1):
        v1 = v1 / beta
        if prec is not None:
            u1 = u1 / beta
        z = u1 if prec is not None else v1
        q = Amul(z)
        alpha = float(z @ q)
        if it > 1:
            q = q - beta * v0
        v0 = q - alpha * v1
        delta = gamma1 * alpha - gamma0 * sigma1 * beta
        rho3 = sigma0 * beta
        rho2 = sigma1 * alpha + gamma0 * gamma1 * beta
        if prec is None:
            beta = float(np.sqrt(v0 @ v0))
        else:
            q = prec(v0)
            beta = float(np.sqrt(v0 @ q))
        rho1 = float(np.hypot(delta, beta))
        if it == 1:
            w0 = z / rho1
        elif it == 2:
            w0 = z / rho1 - (rho2 / rho1) * w1
        else:
            w0 = -(rho3 / rho1) * w0 - (rho2 / rho1) * w1
            w0 = w0 + z / rho1
        gamma0, gamma1 = gamma1, delta / rho1
        x = x + gamma1 * eta * w0
        sigma0, sigma1 = sigma1, beta / rho1
        eta = -sigma1 * eta
        hist.append(abs(eta))
        if abs(eta) <= goal:
            return x, it, True, hist
        if prec is not None:
            u1, q = q, u1
        v0, v1 = v1, v0
        w0, w1 = w1, w0
    return x, max_iter, False, hist
