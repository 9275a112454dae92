"""The AMGe V-cycle as the benchmark runs it.  Hierarchy::Mult in preconditioner mode runs the first call with a
(rhs, sol) buffer pair directly, records the cycle on the second call and replays it afterwards, as a CUDA graph or
as the persistent program kernel (pe_prog.cu); its coarse solver is the device-resident PCG, whose scalars never
leave the GPU.  These tests check that every execution mode computes what the direct cycle computes, for every
smoother, that the mode the test expects is the one that ran (api.Solver.replay_mode), and that the device-resident
PCG follows the same stopping rules as the host PCG and the oracle, indefinite and semidefinite operators included.

Expected execution modes, from the second call with one buffer pair on (the first runs directly: it allocates work
vectors and builds lazy matrix formats; the second records the cycle and launches the recording; later calls replay it):
  * "Use CUDA graph" on (the default): graph;
  * "Use persistent program" on: program when every recorded op has a program implementation (the multicolour SELL
    Gauss-Seidel sweep, SELL/CSR SpMV and the vector ops, PE_OP_* in pe_core.cuh), otherwise the graph, through the
    program -> graph fallback.
The expected mode is part of each test id, so the report lists the mode every configuration ran in."""
import numpy as np
import pytest

from parelag_b200 import api, capi
from oracle import amge, drivers, solve as orc

pytestmark = pytest.mark.gpu

ESS = np.ones(6, dtype=np.int32)


@pytest.fixture(scope="module")
def sess():
    return api.session()


@pytest.fixture(scope="module")
def hier():
    return amge.build_hierarchy((8, 8, 8), 3)[1]


def make_sequence(seqs):
    S = api.Sequence(4, len(seqs))
    for l, s in enumerate(seqs):
        for j in range(4):
            S.set_bdr_mask(l, j, drivers.bdr_mask(s.dof[j]))
            if j < 3:
                S.set_D(l, j, s.D[j])
            if l + 1 < len(seqs):
                S.set_P(l, j, s.P[j])
    return S


class tuning:
    """set capi tuning keys for the duration of a with-block"""

    def __init__(self, **kv):
        self.kv = {getattr(capi, "TUNE_" + k): v for k, v in kv.items()}

    def __enter__(self):
        self.old = {k: capi.get_tuning(k) for k in self.kv}
        for k, v in self.kv.items():
            capi.set_tuning(k, v)

    def __exit__(self, *exc):
        for k, v in self.old.items():
            capi.set_tuning(k, v)


def sell_rows(kernel):
    """TUNE_SELL_MIN_ROWS for the Gauss-Seidel / SpMV kernel family: "sell" forces SELL-C-sigma, "csr" forbids it,
    None keeps the default"""
    return {"sell": 0, "csr": 1 << 30}.get(kernel)


def with_sell(kernel, **kv):
    rows = sell_rows(kernel)
    if rows is not None:
        kv["SELL_MIN_ROWS"] = rows
    return tuning(**kv)


def amge_entries(form, smoother, ordering, damping, omega, cheby, mode, coarse_its=3, coarse_tol=1e-4, hiptmair=None):
    e = drivers.library_entries(form, ordering=ordering, smoother=smoother, damping=damping, omega=omega,
                                cheby_order=cheby, coarse_its=coarse_its, coarse_tol=coarse_tol, hiptmair=hiptmair)
    e["AMGe"][1]["Use CUDA graph"] = mode != "direct"
    e["AMGe"][1]["Use persistent program"] = mode == "program"
    return e


def rhs_sequence(n, marker, count, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        r = rng.standard_normal(n)
        r[marker] = 0.0
        out.append(r)
    return out


def run_prec(sess, solver, rs, b=None, z=None):
    """prec_mult_device on the SAME two device buffers for every right-hand side: outputs and the mode of each call"""
    n = len(rs[0])
    b = capi.Vec(sess, n) if b is None else b
    z = capi.Vec(sess, n) if z is None else z
    outs, modes = [], []
    for r in rs:
        b.upload(r)
        solver.prec_mult_device(b, z)
        outs.append(z.download())
        modes.append(solver.replay_mode())
    return outs, modes


def rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


# ------------------------------------------------------------------------------------------------------------------
# a + b: every smoother, forms 0, 1, 2; direct, graph and program execution of the same preconditioner
# (name, "GS ordering", kernel family, damping, omega, Chebyshev order)
SMOOTHERS = [
    ("Jacobi", "natural", None, 1.0, 1.0, 2),
    ("L1 Jacobi", "natural", None, 1.0, 1.0, 2),
    ("Lumped Jacobi", "natural", None, 1.0, 1.0, 2),
    ("L1 Gauss-Seidel", "natural", "sell", 1.0, 1.0, 2),
    ("L1 Gauss-Seidel", "natural", "csr", 1.0, 1.0, 2),
    ("L1 Gauss-Seidel", "multicolor", "sell", 1.0, 1.0, 2),
    ("L1 Gauss-Seidel", "multicolor", "csr", 1.0, 1.0, 2),
    ("L1 Gauss-Seidel Truncated", "natural", None, 1.0, 1.0, 2),
    ("Gauss-Seidel", "natural", None, 1.0, 1.0, 2),
    ("Gauss-Seidel", "natural", None, 0.9, 1.2, 2),
    ("Chebyshev", "natural", None, 1.0, 1.0, 1),
    ("Chebyshev", "natural", None, 1.0, 1.0, 3),
    ("Hypre Jacobi", "natural", None, 1.0, 1.0, 2),
]


def program_mode(smoother, ordering, kernel):
    """the mode "Use persistent program" runs in: only the multicolour SELL sweep has a program op"""
    return "program" if (smoother, ordering, kernel) == ("L1 Gauss-Seidel", "multicolor", "sell") else "graph"


def _cases():
    out = []
    for form in (0, 1, 2):
        for (name, ordering, kernel, w, om, cheby) in SMOOTHERS:
            # Lumped Jacobi divides by row sums.  Those vanish on the H1 stiffness rows of form 0 and on the
            # auxiliary-space operators D^T A D of Hiptmair, and the cycle overflows.  So it runs on forms 1 and 2
            # as a plain smoother.
            hiptmair = form > 0 and name != "Lumped Jacobi"
            if name == "Lumped Jacobi" and form == 0:
                continue
            pm = program_mode(name, ordering, kernel)
            tag = "%s-%s-%s-w%g-om%g-cheb%d" % (name.replace(" ", ""), ordering, kernel or "default", w, om, cheby)
            out.append(pytest.param(form, hiptmair, name, ordering, kernel, w, om, cheby, pm,
                                    id="form%d%s-%s-program_runs_as_%s" % (form, "-hiptmair" if hiptmair else "", tag, pm)))
    return out


NCALLS = 6


@pytest.mark.parametrize("form,hiptmair,smoother,ordering,kernel,damping,omega,cheby,prog_mode", _cases())
def test_execution_modes_match_direct_and_oracle(sess, hier, form, hiptmair, smoother, ordering, kernel, damping, omega,
                                                 cheby, prog_mode):
    seqs = hier
    A, marker = drivers.system_matrix(seqs[0], form, ESS)
    rs = rhs_sequence(A.shape[0], marker, NCALLS, seed=100 + form)
    S = make_sequence(seqs)
    outs, modes = {}, {}
    with with_sell(kernel):
        for mode in ("direct", "graph", "program"):
            xml = api.library_xml(amge_entries(form, smoother, ordering, damping, omega, cheby, mode, hiptmair=hiptmair))
            solver = api.Solver(xml, "PCG-AMGe", A, S, 0, form, ESS)
            outs[mode], modes[mode] = run_prec(sess, solver, rs)
            solver.free()
    S.free()
    # b: the path that ran.  A failed recording would silently run every call directly.
    assert modes["direct"] == ["direct"] * NCALLS
    assert modes["graph"] == ["direct"] + ["graph"] * (NCALLS - 1)
    assert modes["program"] == ["direct"] + [prog_mode] * (NCALLS - 1)
    # a: a recorded cycle starts from sol = 0 and reads the new right-hand side on every replay.  Call 1 of every
    # solver is direct and builds the lazy matrix formats in all three, so every call index compares the same kernels.
    H = drivers.amge_pcg_solver(seqs, form, ESS, A, ordering=ordering, smoother_type=smoother, damping=damping,
                                omega=omega, cheby_order=cheby, hiptmair=hiptmair)
    # Chebyshev's eigenvalue estimate agrees with the oracle's to 1e-8 only (test_kernels_gpu.py::test_chebyshev)
    tol = 1e-9 if smoother == "Chebyshev" else 1e-11
    for i, r in enumerate(rs):
        zo = H.mult(r)
        assert np.array_equal(outs["graph"][i], outs["direct"][i]), (i, rel(outs["graph"][i], outs["direct"][i]))
        # the program's dot products use another reduction tree (PE_OP_DOT); it differs only in the last bits
        assert np.linalg.norm(outs["program"][i] - outs["direct"][i]) <= 1e-13 * np.linalg.norm(zo), i
        if prog_mode == "graph":
            assert np.array_equal(outs["program"][i], outs["direct"][i]), i
        for mode in outs:
            assert rel(outs[mode][i], zo) <= tol, (mode, i, rel(outs[mode][i], zo))
    # consecutive outputs differ: replays did not return a stale result
    assert all(not np.array_equal(outs["graph"][i], outs["graph"][i + 1]) for i in range(NCALLS - 1))


# ------------------------------------------------------------------------------------------------------------------
# c: two buffer pairs.  Pair A is prec_mult_device's (copy-in, copy-out) pair; pair B is the one the outer PCG's
# device-resident loop passes to its preconditioner: PCG with "Maximum iterations" 2 and zero tolerances applies the
# V-cycle exactly three times.  Sequence: A A A, B B B, A A A.
@pytest.mark.parametrize("mode,kernel,replayed", [("graph", "csr", "graph"), ("graph", "sell", "graph"),
                                                  ("program", "sell", "program")],
                         ids=["graph-csr", "graph-sell", "program-sell"])
def test_buffer_pair_switching_records_again(sess, hier, mode, kernel, replayed):
    seqs = hier
    form = 2
    A, marker = drivers.system_matrix(seqs[0], form, ESS)
    rs = rhs_sequence(A.shape[0], marker, 7, seed=7)
    S = make_sequence(seqs)
    res = {}
    with with_sell(kernel):
        for m in ("direct", mode):
            e = amge_entries(form, "L1 Gauss-Seidel", "multicolor", 1.0, 1.0, 2, m)
            e["PCG-AMGe"][1].update({"Maximum iterations": 2, "Relative tolerance": 0.0, "Absolute tolerance": 0.0})
            solver = api.Solver(api.library_xml(e), "PCG-AMGe", A, S, 0, form, ESS)
            b, z = capi.Vec(sess, A.shape[0]), capi.Vec(sess, A.shape[0])
            o1, m1 = run_prec(sess, solver, rs[:3], b, z)            # A A A
            x = solver.mult(rs[3])                                    # B B B
            hist = solver.history()
            mB = solver.replay_mode()
            o2, m2 = run_prec(sess, solver, rs[4:], b, z)            # A A A
            res[m] = (o1 + o2, m1 + [mB] + m2, x, hist)
            solver.free()
    S.free()
    assert res["direct"][1] == ["direct"] * 7
    # B's third call replays B's graph; A's graph was displaced, so A is warmed (direct) and recorded again
    assert res[mode][1] == ["direct", replayed, replayed, replayed, "direct", replayed, replayed]
    assert len(res[mode][3][0]) == 3 and res[mode][3][1] == 2
    if mode == "graph":
        for o, od in zip(res[mode][0], res["direct"][0]):
            assert np.array_equal(o, od)
        assert np.array_equal(res[mode][2], res["direct"][2])
        assert np.array_equal(res[mode][3][0], res["direct"][3][0])
    else:
        for o, od in zip(res[mode][0], res["direct"][0]):
            assert np.linalg.norm(o - od) <= 1e-13 * np.linalg.norm(od)
        assert rel(res[mode][2], res["direct"][2]) <= 1e-12
    H = drivers.amge_pcg_solver(seqs, form, ESS, A, ordering="multicolor")
    for o, r in zip(res[mode][0], rs[:3] + rs[4:]):
        assert rel(o, H.mult(r)) <= 1e-11


# ------------------------------------------------------------------------------------------------------------------
# d: programmatic dependent launch inside a replayed graph, at 32^3 (about 101 k H(div) rows: kernels with many CTAs).
# Bit-identity is the contract (DESIGN.md section 4): every kernel reads its predecessor's output after
# griddepcontrol.wait.  The oracle's Python Coarsen() is too slow at this size.
@pytest.mark.parametrize("smoother,ordering,kernel", [("L1 Gauss-Seidel", "multicolor", "sell"),
                                                      ("L1 Gauss-Seidel", "multicolor", "csr"),
                                                      ("L1 Jacobi", "natural", "sell")],
                         ids=["gs-multicolor-sell", "gs-multicolor-csr", "l1jacobi-sell"])
def test_pdl_in_replayed_graph_is_bit_identical(sess, smoother, ordering, kernel):
    form, ncalls = 2, 12          # calls 3..12: ten replays
    S = api.Sequence.hex((32, 32, 32), 3)
    outs, modes = {}, {}
    with with_sell(kernel):
        for arm, mode, pdl in (("direct", "direct", 1), ("graph-pdl1", "graph", 1), ("graph-pdl0", "graph", 0)):
            with tuning(PDL=pdl):
                A = S.assemble_system(sess, 0, form, ESS)
                n = A.info()[0]
                if arm == "direct":
                    rs = rhs_sequence(n, np.zeros(n, dtype=bool), ncalls, seed=32)
                xml = api.library_xml(amge_entries(form, smoother, ordering, 1.0, 1.0, 2, mode))
                solver = api.Solver(xml, "PCG-AMGe", A, S, 0, form, ESS)
                outs[arm], modes[arm] = run_prec(sess, solver, rs)
                solver.free()
    S.free()
    assert n > 100000
    assert modes["direct"] == ["direct"] * ncalls
    for arm in ("graph-pdl1", "graph-pdl0"):
        assert modes[arm] == ["direct"] + ["graph"] * (ncalls - 1), arm
        for i in range(ncalls):
            assert np.array_equal(outs[arm][i], outs["direct"][i]), (arm, i, rel(outs[arm][i], outs["direct"][i]))
    assert np.all(np.isfinite(outs["direct"][-1])) and np.linalg.norm(outs["direct"][-1]) > 0


# ------------------------------------------------------------------------------------------------------------------
# e: the device-resident PCG ("Maximum iterations" <= 10, "Print level" -1) against the host PCG ("Print level" 0,
# the loop of KrylovSolver::Mult) and the oracle (mfem::CGSolver::Mult restated)
def pcg_lib(max_iter, rtol, atol, device, prec):
    k = {"Solver name": "PCG", "Print level": -1 if device else 0, "Maximum iterations": max_iter,
         "Relative tolerance": float(rtol), "Absolute tolerance": float(atol)}
    lib = {"K": ("Krylov", k)}
    if prec is not None:
        lib["P"] = ("Hypre", {"Type": prec, "Sweeps": 1, "Damping Factor": 1.0})
        k["Preconditioner"] = "P"
    return api.library_xml(lib)


def oracle_prec(A, prec):
    if prec is None:
        return None
    So = orc.Smoother(A, type=drivers.SMOOTHER_TYPES[prec])
    return lambda r: So.apply(r, np.zeros_like(r), False)


def pcg_dens(A, prec, b, max_iter):
    """(Ad, d) of each check of mfem::CGSolver::Mult with zero tolerances (plain numpy; used to certify that an
    operator gives the sign the case is about)"""
    M = (lambda r: r.copy()) if prec is None else prec
    r = b.copy(); z = M(r); d = z.copy(); nom = d @ r
    dens = []
    for i in range(max_iter):
        z = A @ d; den = d @ z; dens.append(den)
        if den == 0:
            break
        alpha = nom / den
        r = r - alpha * z
        z = M(r); betanom = r @ z
        d = z + betanom / nom * d
        nom = betanom
    return dens


def check_pcg(A, b, max_iter, rtol, atol, prec=None, x0=None):
    """device path, host path and oracle agree: x, history, iteration count, convergence flag"""
    xo, ito, convo, histo = orc.pcg(A, oracle_prec(A, prec), b, rtol=rtol, atol=atol, max_iter=max_iter, x0=x0)
    histo = np.array(histo)
    got = {}
    for device in (True, False):
        solver = api.Solver(pcg_lib(max_iter, rtol, atol, device, prec), "K", A, None, 0, 0, None)
        x = solver.mult(b, x0=x0)
        got[device] = (x, *solver.history())
        solver.free()
    scale = max(np.linalg.norm(xo), np.linalg.norm(b))
    for device, (x, hist, it, conv) in got.items():
        where = "device" if device else "host"
        assert (it, conv) == (ito, convo), (where, it, conv, ito, convo)
        assert len(hist) == len(histo), (where, hist, histo)
        assert np.all(np.abs(hist - histo) <= 1e-13 * np.maximum(np.abs(histo), np.abs(histo[0]) * 1e-3)), (where, hist, histo)
        assert np.linalg.norm(x - xo) <= 1e-13 * scale, (where, np.linalg.norm(x - xo) / scale)
    return ito, convo, histo


@pytest.fixture(scope="module")
def spd(hier):
    A, marker = drivers.system_matrix(hier[0], 0, ESS)
    b = np.random.default_rng(41).standard_normal(A.shape[0])
    b[marker] = 0.0
    return A, b


@pytest.mark.parametrize("prec", [None, "L1 Jacobi"])
def test_device_pcg_stops_at_every_iteration(sess, spd, prec):
    """Relative tolerance between consecutive history values, so that betanom < r0 first holds at iteration k"""
    A, b = spd
    hist = np.array(orc.pcg(A, oracle_prec(A, prec), b, rtol=0.0, atol=0.0, max_iter=10)[3])
    hit = []
    for k in range(1, 11):
        above = hist[1:k].min() if k > 1 else hist[0]
        if not hist[k] < above * (1 - 1e-6):
            continue                                  # (B r, r) is not monotone: k cannot be the first to fall below
        r0 = np.sqrt(hist[k] * above)
        it, conv, _ = check_pcg(A, b, 10, np.sqrt(r0 / hist[0]), 0.0, prec)
        assert (it, conv) == (k, True)
        hit.append(k)
    assert len(hit) >= 8, hit


@pytest.mark.parametrize("prec", [None, "L1 Jacobi"])
def test_device_pcg_limits_and_tolerances(sess, spd, prec):
    A, b = spd
    # converged at iteration 0: zero right-hand side, and an absolute tolerance above the initial norm
    assert check_pcg(A, np.zeros_like(b), 5, 1e-6, 1e-6, prec)[:2] == (0, True)
    h0 = check_pcg(A, b, 5, 0.0, 0.0, prec)[2][0]
    assert check_pcg(A, b, 5, 0.0, 2.0 * np.sqrt(h0), prec)[:2] == (0, True)
    # iteration limit 1 and 10
    for m in (1, 10):
        assert check_pcg(A, b, m, 0.0, 0.0, prec)[:2] == (m, False)
    # absolute tolerance only, relative tolerance only (stop at 4 from the zero-tolerance history)
    hist = check_pcg(A, b, 10, 0.0, 0.0, prec)[2]
    it, conv, _ = check_pcg(A, b, 10, 0.0, np.sqrt(np.sqrt(hist[4] * hist[1:4].min())), prec)
    assert conv and 1 <= it <= 4
    it, conv, _ = check_pcg(A, b, 10, np.sqrt(np.sqrt(hist[4] * hist[1:4].min()) / hist[0]), 0.0, prec)
    assert conv and 1 <= it <= 4
    # iterative_mode: the initial guess starts the iteration
    x0 = np.random.default_rng(5).standard_normal(len(b))
    check_pcg(A, b, 6, 1e-3, 0.0, prec, x0=x0)


def tridiag(diag, off):
    import scipy.sparse as sp
    n = len(diag)
    return sp.diags([np.full(n - 1, off), diag, np.full(n - 1, off)], [-1, 0, 1], format="csr")


def test_device_pcg_indefinite_and_semidefinite(sess):
    """mfem::CGSolver::Mult: a negative (Ad, d) goes on with a negative step; only an exact zero stops, unconverged,
    at the iteration that computed it; a negative initial (B r, r) stops at once"""
    n = 64
    # negative (Ad, d) at the first check
    A = tridiag(np.where(np.arange(n) < 48, -3.0, 1.0) + 0.01 * np.arange(n), 0.5)
    b = np.ones(n)
    dens = pcg_dens(A, None, b, 6)
    assert dens[0] < 0
    it, conv, hist = check_pcg(A, b, 6, 0.0, 0.0)
    assert (it, conv, len(hist)) == (6, False, 7)
    # positive at the first check, negative later
    A = tridiag(np.where(np.arange(n) % 4 == 0, -0.6, 2.0) + 0.01 * np.arange(n), 0.3)
    b = np.linspace(1.0, 2.0, n)
    dens = pcg_dens(A, None, b, 8)
    assert dens[0] > 0 and min(dens) < 0, dens
    it, conv, hist = check_pcg(A, b, 8, 0.0, 0.0)
    assert (it, conv, len(hist)) == (8, False, 9)
    # (Ad, d) == 0 at the first check: b in the null space of a semidefinite A
    import scipy.sparse as sp
    A = sp.diags(np.where(np.arange(n) % 2 == 0, 1.0, 0.0), format="csr")
    b = np.where(np.arange(n) % 2 == 1, 1.0, 0.0)
    it, conv, hist = check_pcg(A, b, 5, 0.0, 0.0)
    assert (it, conv, list(hist)) == (0, False, [n / 2])
    # (Ad, d) == 0 in iteration 1 (exact arithmetic): d_1 = r_1 + d_0 lies in the null space; final_iter = 2
    b = np.ones(n)
    assert pcg_dens(A, None, b, 3) == [n / 2, 0.0]
    it, conv, hist = check_pcg(A, b, 5, 0.0, 0.0)
    assert (it, conv, list(hist)) == (2, False, [float(n), float(n)])
    # negative initial (B r, r): a Jacobi preconditioner of a negative diagonal
    A = tridiag(-2.0 - 0.01 * np.arange(n), 0.5)
    it, conv, hist = check_pcg(A, np.ones(n), 5, 1e-6, 0.0, prec="Jacobi")
    assert (it, conv, len(hist)) == (0, False, 1) and hist[0] < 0


# the SPD cases once more, as the coarse solver of a 2-level hierarchy replayed as a graph and as the program:
# PE_OP_PCG_STEP, PE_OP_AXPY_DEV and PE_OP_XPBY_DEV inside the recorded cycle
@pytest.mark.parametrize("coarse_its,coarse_tol", [(1, 0.0), (2, 1e-2), (3, 1e-4), (5, 1e-6), (10, 0.0), (10, 1e-3)])
def test_coarse_pcg_in_recorded_cycle(sess, hier, coarse_its, coarse_tol):
    seqs = hier[:2]
    form = 2
    A, marker = drivers.system_matrix(seqs[0], form, ESS)
    rs = rhs_sequence(A.shape[0], marker, 5, seed=coarse_its)
    S = make_sequence(seqs)
    outs, modes = {}, {}
    with with_sell("sell"):
        for mode in ("direct", "graph", "program"):
            e = amge_entries(form, "L1 Gauss-Seidel", "multicolor", 1.0, 1.0, 2, mode, coarse_its=coarse_its,
                             coarse_tol=coarse_tol)
            solver = api.Solver(api.library_xml(e), "PCG-AMGe", A, S, 0, form, ESS)
            assert solver.num_levels() == 2
            outs[mode], modes[mode] = run_prec(sess, solver, rs)
            solver.free()
    S.free()
    assert modes["graph"][2:] == ["graph"] * 3 and modes["program"][2:] == ["program"] * 3
    H = drivers.amge_pcg_solver(seqs, form, ESS, A, ordering="multicolor", coarse_its=coarse_its, coarse_tol=coarse_tol)
    for i, r in enumerate(rs):
        zo = H.mult(r)
        assert np.array_equal(outs["graph"][i], outs["direct"][i]), i
        assert np.linalg.norm(outs["program"][i] - outs["direct"][i]) <= 1e-13 * np.linalg.norm(zo), i
        for mode in outs:
            assert rel(outs[mode][i], zo) <= 1e-11, (mode, i)
