"""Time SetOperator on the benchmark's solver against a new BuildSolver (one B200).

configs[1] at --size^3 as bench.py builds it (H(div), PCG with the AMGe auxiliary-space preconditioner, Hiptmair with
multicolour l1-Gauss-Seidel): BuildSolver(A1); SetOperator(A2) with A2 = S A1 S (S a seeded positive diagonal, 1 on the
essential rows); the two direct V-cycles that follow (the second records the cycle) and one replayed V-cycle; then
BuildSolver(A2) for comparison.  The card name and power limit go into the same JSON (--out).  Every time is a host
clock around work that ends in a device synchronise.

The split of SetOperator comes from its phase timers (TimeManager: Galerkin products, Hiptmair auxiliary operators,
smoothers and coarse solver, colour-numbered copies).  The fine-level numeric product P^T A P (pe_rap_numeric, P the
level-1 prolongator ComputeTrueP) is also timed on its own, with its two parts: the two-pass A P and the numeric
P^T (A P) into A_1's pattern.  Bytes are computed from the shapes, each array read or written once (int32 indices,
FP64 values): A P reads A and P and writes A P; P^T (A P) reads P^T and A P, the row pointers and columns of A_1, and
writes A_1's values.

--config darcy / spe10: the mixed solver bench.py --config darcy / spe10 builds (configs[1] MultigridTestDarcy at 136^3 with
4 levels, configs[3] SPE10-shaped 60 x 220 x 85 with the synthetic lognormal permeability; --mixed-solver ldu: GMRES +
Block LDU with AMGe V-cycles on M and on the Schur complement, blocked: GMRES + the blocked AMGe hierarchy with Block
Jacobi smoothers; multicolour ordering).  BuildSolver(M1, B, Bt); SetOperator(M2, B, Bt) with M2 = S M1 S (S a seeded
positive diagonal); the first GMRES solve after the update; then BuildSolver(M2, B, Bt) and its first GMRES solve.  The
update's phase timers nest: "block inverses" (the A00 and S inverses, for Block LDU the inner AMGe hierarchies with
their own Galerkin products and smoothers) and "Schur complements" run inside "smoothers and coarse solver" of a blocked
hierarchy."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from parelag_b200 import api, capi  # noqa: E402
import bench  # noqa: E402


def sync(ctx):
    capi.lib().pe_ctx_sync(ctx.h)


def timed(ctx, f):
    sync(ctx)
    t0 = time.perf_counter()
    out = f()
    sync(ctx)
    return time.perf_counter() - t0, out


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in q.split(",")]
        return name, limit
    except Exception as e:     # the numbers are still written, marked as unattributed
        return "unknown (%s)" % e, "unknown"


PHASES = ("Galerkin products", "Hiptmair auxiliary operators", "smoothers and coarse solver", "colour-numbered copies")


def csr_bytes(rows, nnz, values=True):
    return 4.0 * (rows + 1) + (12.0 if values else 4.0) * nnz


def fine_rap(ctx, S, A1, A2, ess, repeats=5):
    """pe_rap_numeric on the fine level alone, and its two parts; best of `repeats`, bytes from the shapes"""
    dA1, dA2 = capi.Mat.from_scipy(ctx, A1), capi.Mat.from_scipy(ctx, A2)
    P = S.true_operator(ctx, 0, "P", 2, ess)
    Pt = P.transpose()
    Ac = capi.rap(ctx, dA1, P)
    AP = capi.spgemm(ctx, dA2, P)
    n, nc = A1.shape[0], P.info()[1]
    nnzA, nnzP, nnzAP, nnzAc = A1.nnz, P.info()[3], AP.info()[3], Ac.info()[3]
    vx, vy = capi.Vec(ctx, n), capi.Vec(ctx, nc)
    vx.upload(np.ones(n))
    P.spmv_t(vx, vy)          # caches P^T on P, as the V-cycle does before an update

    def best(f):
        f()
        return min(timed(ctx, f)[0] for _ in range(repeats))

    def two_pass():
        m = capi.spgemm(ctx, dA2, P)
        m.free()
    t_rap = best(lambda: capi.rap_numeric(ctx, dA2, P, Ac))
    t_ap = best(two_pass)
    t_num = best(lambda: capi.spgemm_numeric(ctx, Pt, AP, Ac))
    b_ap = csr_bytes(n, nnzA) + csr_bytes(n, nnzP) + csr_bytes(n, nnzAP)
    b_num = csr_bytes(nc, nnzP) + csr_bytes(n, nnzAP) + csr_bytes(nc, nnzAc, values=False) + 8.0 * nnzAc
    out = {"rows": n, "cols": nc, "nnz_A": int(nnzA), "nnz_P": int(nnzP), "nnz_AP": int(nnzAP), "nnz_Ac": int(nnzAc),
           "rap_numeric_s": t_rap, "rap_numeric_bytes": b_ap + b_num, "rap_numeric_GBps": (b_ap + b_num) / t_rap / 1e9,
           "AP_two_pass_s": t_ap, "AP_bytes": b_ap, "AP_GBps": b_ap / t_ap / 1e9,
           "PtAP_numeric_s": t_num, "PtAP_numeric_bytes": b_num, "PtAP_numeric_GBps": b_num / t_num / 1e9}
    for m in (dA1, dA2, P, Pt, Ac, AP):
        m.free()
    vx.free(); vy.free()
    return out


MIXED_PHASES = ("Galerkin products", "Schur complements", "block inverses", "smoothers and coarse solver")


def mixed(ctx, args):
    """--config darcy / spe10: SetOperator(M2, B, Bt) against BuildSolver on the same blocks, and the first GMRES solve"""
    if args.config == "darcy":
        S = api.Sequence.hex((136,) * 3, 4, jstart=2)
        shape = {"size": 136, "levels": 4}
    else:
        dims, Lspe = (60, 220, 85), (1200.0, 2200.0, 170.0)
        kinv = 10.0 ** (-np.clip(np.random.default_rng(13).normal(-1.0, 1.5, size=dims[0] * dims[1] * dims[2]), -4.0, 2.0))
        S = api.Sequence.hex(dims, 4, L=Lspe, beta=kinv, jstart=2)
        shape = {"dims": list(dims), "levels": 4}
    Md, Bd, Btd = S.assemble_darcy(ctx, 0)
    M1, B, Bt = Md.to_scipy(), Bd.to_scipy(), Btd.to_scipy()
    for m in (Md, Bd, Btd):
        m.free()
    rows = np.repeat(np.arange(M1.shape[0]), np.diff(M1.indptr))
    sc = np.random.default_rng(1).uniform(0.5, 2.0, M1.shape[0])
    M2 = M1.copy()
    M2.data = M1.data * sc[rows] * sc[M1.indices]
    if args.mixed_solver == "ldu":
        xml, name, ess = api.library_xml(bench.library_darcy_ldu("multicolor")), "GMRES with Block LDU", np.zeros((2, 6), dtype=np.int32)
    else:
        xml, name, ess = api.library_xml(bench.library_darcy("multicolor")), "GMRES with blocked AMGe", None
    n = M1.shape[0] + B.shape[0]
    b = np.random.default_rng(2).standard_normal(n)
    vb, vz = capi.Vec(ctx, data=b), capi.Vec(ctx, n)
    res = dict(shape, config=args.config, solver=name, rows_M=int(M1.shape[0]), nnz_M=int(M1.nnz), rows_B=int(B.shape[0]),
               nnz_B=int(B.nnz))

    def blocks(M):
        return [[capi.Mat.from_scipy(ctx, M), capi.Mat.from_scipy(ctx, Bt)], [capi.Mat.from_scipy(ctx, B), None]]
    m1 = blocks(M1)
    res["build_solver_M1_s"], solver = timed(ctx, lambda: api.BlockSolver(xml, name, m1, S, 0, [2, 3], ess_attr=ess))
    for _ in range(3):
        solver.prec_mult_device(vb, vz)
    m2 = blocks(M2)
    api.lib().pe_api_timer_clear()
    res["set_operator_M2_s"], _ = timed(ctx, lambda: solver.set_blocks(m2))
    res["set_operator_phases_s"] = {k: api.timer("SetOperator: " + k) for k in MIXED_PHASES}
    res["first_solve_after_update_s"], x_upd = timed(ctx, lambda: solver.mult(b))
    h_upd = solver.history()
    solver.free()
    m2b = blocks(M2)
    res["build_solver_M2_s"], fresh = timed(ctx, lambda: api.BlockSolver(xml, name, m2b, S, 0, [2, 3], ess_attr=ess))
    res["first_solve_fresh_s"], x_fresh = timed(ctx, lambda: fresh.mult(b))
    h_fresh = fresh.history()
    fresh.free()
    res["gmres_iterations_update_fresh"] = [h_upd[1], h_fresh[1]]
    res["fresh_equals_update"] = bool(np.array_equal(x_upd, x_fresh) and np.array_equal(h_upd[0], h_fresh[0]))
    vb.free(); vz.free()
    S.free()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="hdiv", choices=["hdiv", "darcy", "spe10"])
    ap.add_argument("--mixed-solver", default="ldu", choices=["ldu", "blocked"], help="darcy / spe10, as bench.py")
    ap.add_argument("--size", type=int, default=144)
    ap.add_argument("--levels", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = api.session()
    if args.config != "hdiv":
        res = mixed(ctx, args)
        res["card"], res["power_limit"] = card()
        line = json.dumps(res)
        print(line)
        if args.out:
            with open(args.out, "w") as f:
                f.write(line + "\n")
        return
    ESS = np.ones(6, dtype=np.int32)
    S = api.Sequence.hex((args.size,) * 3, args.levels, jstart=1)
    xml = api.library_xml(bench.library("multicolor", 2))
    name = "PCG with Auxiliary Space Preconditioner"
    A1 = S.assemble_system(ctx, 0, 2, ESS).to_scipy()
    marker = np.zeros(A1.shape[0], dtype=bool)
    rows = np.repeat(np.arange(A1.shape[0]), np.diff(A1.indptr))
    unit = (A1.indices == rows) & (A1.data == 1.0)
    offdiag_nz = np.bincount(rows[(A1.indices != rows) & (A1.data != 0.0)], minlength=A1.shape[0])
    marker[rows[unit]] = offdiag_nz[rows[unit]] == 0      # eliminated rows: unit diagonal, nothing else
    s = np.random.default_rng(1).uniform(0.5, 2.0, A1.shape[0])
    s[marker] = 1.0
    A2 = A1.copy()
    A2.data = A1.data * s[rows] * s[A1.indices]
    b = np.random.default_rng(2).standard_normal(A1.shape[0])
    b[marker] = 0.0
    vb, vz = capi.Vec(ctx, data=b), capi.Vec(ctx, A1.shape[0])
    res = {"size": args.size, "levels": args.levels, "rows": int(A1.shape[0]), "nnz": int(A1.nnz)}

    res["fine_galerkin_product"] = fine_rap(ctx, S, A1, A2, ESS)

    m1 = capi.Mat.from_scipy(ctx, A1)
    res["build_solver_A1_s"], solver = timed(ctx, lambda: api.Solver(xml, name, m1, S, 0, 2, ESS))
    solver.prec_mult_device(vb, vz)
    solver.prec_mult_device(vb, vz)
    solver.prec_mult_device(vb, vz)
    res["replay_mode_before"] = solver.replay_mode()
    m2 = capi.Mat.from_scipy(ctx, A2)
    res["set_operator_A2_s"], _ = timed(ctx, lambda: solver.set_operator(m2))
    res["set_operator_phases_s"] = {k: api.timer("SetOperator: " + k) for k in PHASES}
    calls = []
    for _ in range(3):
        t, _ = timed(ctx, lambda: solver.prec_mult_device(vb, vz))
        calls.append((t, solver.replay_mode()))
    res["after_update_calls"] = [{"s": t, "mode": m} for t, m in calls]
    z_upd = vz.download()
    solver.free()

    m2b = capi.Mat.from_scipy(ctx, A2)
    res["build_solver_A2_s"], fresh = timed(ctx, lambda: api.Solver(xml, name, m2b, S, 0, 2, ESS))
    for _ in range(3):
        fresh.prec_mult_device(vb, vz)
    res["fresh_equals_update"] = bool(np.array_equal(vz.download(), z_upd))
    n1 = fresh.level_info(1)
    fresh.free()
    res["level1_rows_nnz_nnzP"] = [int(x) for x in n1]
    res["card"], res["power_limit"] = card()
    S.free()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
