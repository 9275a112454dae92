#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native AMGe solve-and-coarsen path.

Metric (BASELINE.json): DOFs/s per V-cycle (+ setup seconds, SpMV/smoother HBM GB/s vs
peak).  Workload at N=1 (configs[1], "MultigridTest2Form"): H(div) problem
A = M_2 + D_2^T M_3 D_2 on the unit cube with n^3 hexahedra (n = 144 -> 9 020 160 RT0
dofs), 5-level AMGe hierarchy built by DeRhamSequence::Coarsen(), Hiptmair smoother
(l1-Gauss-Seidel on the H(div) operator and on D^T A D in H(curl)), coarse solver
"PCG-GS" (3 PCG iterations preconditioned by the same smoother), all boundary
attributes essential.  A step = one application of the AMGe V-cycle
(Hierarchy::Mult) to a device-resident residual.

  python bench.py --gpus N --steps K --warmup W            (this implementation)
  python bench.py --impl reference --gpus N --steps K ...  (CPU reference arm)

N > 1: one process per GPU (torchrun), one mesh box per GPU -- BASELINE configs[4], examples/3DHdivWeakScaling.cpp:
the unit cube cut into 2x1x1, 2x2x1, 2x2x2 boxes of n^3 hexahedra each, vertices moved by y += exp(z)/2,
x += sin(y) (trilinear hexahedra, :148-158), essential data on boundary attributes 2-5, natural on 1 and 6
(:53-66).  Every rank coarsens its own box, the levels are glued by SharingMaps, and the V-cycle exchanges the
ParCSR halo over NVLink peer memory (or NCCL send/recv).  Weak scaling: per-GPU work is fixed,
value = global dofs / max-over-ranks time.

Before anything is timed, at every N, a `parity` block checks the product against the oracle (tests/parity_checks.py):
N = 1: Coarsen + V-cycle + PCG history on a small mesh, and one SpMV and one multicolour Gauss-Seidel sweep of the
FULL-SIZE fine operator against oracle/solve_oracle.c; N > 1: the box-decomposed hierarchy (same geometry, 4^3
hexahedra per box) against the oracle's single-domain hierarchy.  The oracle is only the checker there.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "vcycle_dofs_per_s"
UNIT = "DOFs/s"
ESS = np.ones(6, dtype=np.int32)
DUMP_MAX_BYTES = 64 * 10 ** 6          # --dump-outputs: all files of one run together


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def library(ordering, form=2):
    """ParameterList 'Preconditioner Library' of examples/testing_helpers/Create2FormParameterList.hpp
    with the coarse solver replaced by the hot-path-only PCG-GS (SURVEY fact 9)."""
    hyp = ("Hypre", {"Type": "L1 Gauss-Seidel", "Sweeps": 1, "Damping Factor": 1.0, "Omega": 1.0,
                     "Cheby Poly Order": 2, "Cheby Poly Fraction": 0.3, "GS ordering": ordering})
    return {
        "Gauss-Seidel": hyp,
        "Hiptmair-GS-GS": ("Hiptmair", {"Primary Smoother": "Gauss-Seidel", "Auxiliary Smoother": "Gauss-Seidel"}),
        "PCG-GS": ("Krylov", {"Solver name": "PCG", "Preconditioner": "Hiptmair-GS-GS", "Print level": -1,
                              "Maximum iterations": 3, "Relative tolerance": 1e-4, "Absolute tolerance": 1e-4}),
        "AMGe-HIP-GS_2": ("AMGe", {"Maximum levels": -1, "Forms": [form], "PreSmoother": "Hiptmair-GS-GS",
                                   "PostSmoother": "Hiptmair-GS-GS", "Coarse solver": "PCG-GS",
                                   "Cycle type": "V-cycle"}),
        "PCG with Auxiliary Space Preconditioner": (
            "Krylov", {"Solver name": "PCG", "Preconditioner": "AMGe-HIP-GS_2", "Print level": -1,
                       "Maximum iterations": 300, "Relative tolerance": 1e-6, "Absolute tolerance": 1e-6}),
    }


def library_h1(ordering):
    """examples/testing_helpers/Create0FormParameterList.hpp with the hot-path-only coarse solver (SURVEY fact 9)"""
    hyp = ("Hypre", {"Type": "L1 Gauss-Seidel", "Sweeps": 1, "Damping Factor": 1.0, "Omega": 1.0, "GS ordering": ordering})
    return {
        "Gauss-Seidel": hyp,
        "PCG-GS": ("Krylov", {"Solver name": "PCG", "Preconditioner": "Gauss-Seidel", "Print level": -1, "Maximum iterations": 3,
                              "Relative tolerance": 1e-4, "Absolute tolerance": 1e-4}),
        "AMGe-GS_0": ("AMGe", {"Maximum levels": -1, "Forms": [0], "PreSmoother": "Gauss-Seidel", "PostSmoother": "Gauss-Seidel",
                               "Coarse solver": "PCG-GS", "Cycle type": "V-cycle"}),
        "PCG with Auxiliary Space Preconditioner": (
            "Krylov", {"Solver name": "PCG", "Preconditioner": "AMGe-GS_0", "Print level": -1, "Maximum iterations": 300,
                       "Relative tolerance": 1e-6, "Absolute tolerance": 1e-6}),
    }


def library_darcy(ordering):
    """examples/example_parameterlists/darcy_example_parameters.xml: GMRES(50) preconditioned by the blocked AMGe
    (Forms 2 3) with a Block Jacobi smoother (A00: l1-GS, S = -(B diag(M)^-1 B^T): l1-GS); coarse solver GMRES + the same"""
    gs = ("Hypre", {"Type": "L1 Gauss-Seidel", "Sweeps": 1, "Damping Factor": 1.0, "Omega": 1.0, "GS ordering": ordering})
    return {
        "Gauss-Seidel": gs,
        "Blk": ("Block Jacobi", {"A00 Inverse": "Gauss-Seidel", "A11 Inverse": "Gauss-Seidel", "Alpha": 1.0, "S Type": "Diagonal"}),
        "GMRES-Blk": ("Krylov", {"Solver name": "GMRES", "Preconditioner": "Blk", "Print level": -1, "Maximum iterations": 5,
                                 "Relative tolerance": 1e-4, "Absolute tolerance": 1e-4, "Restart size": 50}),
        "AMGe-Blk": ("AMGe", {"Maximum levels": -1, "Forms": [2, 3], "PreSmoother": "Blk", "PostSmoother": "Blk",
                              "Coarse solver": "GMRES-Blk", "Cycle type": "V-cycle"}),
        "GMRES with blocked AMGe": ("Krylov", {"Solver name": "GMRES", "Preconditioner": "AMGe-Blk", "Print level": -1,
                                               "Maximum iterations": 300, "Relative tolerance": 1e-6, "Absolute tolerance": 1e-6,
                                               "Restart size": 50}),
    }


def library_darcy_ldu(ordering):
    """examples/example_parameterlists/spe10_example_parameters.xml: GMRES(50) preconditioned by Block LDU whose A00
    inverses are AMGe V-cycles on the H(div) mass block (Forms 2) and whose Schur-complement inverse is an AMGe V-cycle
    on S = -(B diag(M)^-1 B^T) (Forms 3) -- the file's BoomerAMG inverses replaced by the hot-path solvers (SURVEY fact 9)"""
    gs = ("Hypre", {"Type": "L1 Gauss-Seidel", "Sweeps": 1, "Damping Factor": 1.0, "Omega": 1.0, "GS ordering": ordering})
    pcg = ("Krylov", {"Solver name": "PCG", "Preconditioner": "Gauss-Seidel", "Print level": -1, "Maximum iterations": 3,
                      "Relative tolerance": 1e-4, "Absolute tolerance": 1e-4})
    amge = lambda form: ("AMGe", {"Maximum levels": -1, "Forms": [form], "PreSmoother": "Gauss-Seidel", "PostSmoother": "Gauss-Seidel",
                                  "Coarse solver": "PCG-GS", "Cycle type": "V-cycle"})
    return {
        "Gauss-Seidel": gs, "PCG-GS": pcg, "AMGe-GS_2": amge(2), "AMGe-GS_3": amge(3),
        "Block-LDU-AMGe": ("Block LDU", {"Damping Factor": 0.775, "A00_1 Inverse": "AMGe-GS_2", "A00_2 Inverse": "AMGe-GS_2",
                                         "A00_3 Inverse": "AMGe-GS_2", "Alpha": 1.0, "S Type": "Diagonal", "S Inverse": "AMGe-GS_3"}),
        "GMRES with Block LDU": ("Krylov", {"Solver name": "GMRES", "Preconditioner": "Block-LDU-AMGe", "Print level": -1,
                                            "Maximum iterations": 300, "Relative tolerance": 1e-6, "Absolute tolerance": 1e-6,
                                            "Restart size": 50}),
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(device), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


def dump_outputs(dirname, arrays, budget=DUMP_MAX_BYTES):
    """--dump-outputs: each array as dirname/<name>.npy in float64.  An array larger than its share of the budget is
    stored at a fixed, seeded sample of its indices (ascending), so two builds run with the same arguments store the same
    entries and can be compared file by file."""
    os.makedirs(dirname, exist_ok=True)
    share = budget // max(len(arrays), 1)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float64).ravel()
        cap = (share - 128) // a.itemsize                  # 128 bytes: the .npy header of a 1-D array
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(2024).choice(a.size, cap, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


def traffic_from_profiles():
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        return json.load(open(p))
    return {}


# ----------------------------------------------------------------------------------------------
# CPU reference / baseline leg (the ONLY place bench.py touches oracle/)
# ----------------------------------------------------------------------------------------------
def cpu_vcycle_setup(n_sample, levels, ranks, hier_from):
    """Oracle V-cycle (oracle/solve.py: hypre/MFEM arithmetic restated in C) on a bounded sample of
    the workload: the same H(div) problem on n_sample^3 hexahedra.  hier_from(n, levels) returns the
    level operators (A0, [P_l], [D_l]) -- inputs of the solve path, not part of what is timed."""
    from oracle import solve as orc
    A0, Ps, Ds = hier_from(n_sample, levels)
    nl = len(Ps) + 1

    def smoother(l, Al):
        kw = lambda M: dict(type=2, ranks=ranks)
        return orc.Hiptmair(Al, Ds[l], kw, kw)

    def coarse(Ac):
        S = smoother(nl - 1, Ac)
        return lambda b, x: orc.pcg(Ac, lambda r: S.apply(r, np.zeros_like(r), False), b, rtol=1e-4, atol=1e-4,
                                    max_iter=3)[0]
    H = orc.build_hierarchy(A0, Ps, smoother, coarse)
    return H, A0.shape[0]


def oracle_hierarchy_inputs(n, levels):
    """Level operators from the oracle's own coarsening (CPU only; small n) -- used by the reference
    arm when no GPU is involved at all."""
    from oracle import amge, drivers
    mesh, seqs = amge.build_hierarchy((n, n, n), levels, jstart=1)
    A, _ = drivers.system_matrix(seqs[0], 2, ESS)
    Ps = [seqs[l].get_P(2, ESS) for l in range(levels - 1)]
    Ds = [seqs[l].get_D(1, ESS) for l in range(levels)]
    return A, Ps, Ds


def time_cpu_vcycles(H, n, steps, warmup, budget_s=25.0):
    rng = np.random.default_rng(0)
    r = rng.standard_normal(n)
    for _ in range(warmup):
        H.mult(r)
    ts = []
    t_all = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        z = H.mult(r)
        ts.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s:
            break
    return float(np.mean(ts)), len(ts), z


def host_threads():
    """threads this process may really use (affinity / cgroup aware)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def host_memory_gb():
    """memory this node offers all ranks together: MemTotal, or the cgroup limit when that is lower.  A constant of the
    box (not MemAvailable), so every rank and both arms of the bench derive the same box size from it."""
    total = 0.0
    try:
        total = int([l for l in open("/proc/meminfo") if l.startswith("MemTotal")][0].split()[1]) / 1048576.0
    except Exception:
        return 0.0
    for f in ("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory/memory.limit_in_bytes"):
        try:
            v = open(f).read().strip()
            if v.isdigit() and 0 < int(v) < (1 << 60):
                total = min(total, int(v) / float(1 << 30))
        except Exception:
            pass
    return total


def fit_box_size(n, world, per_rank_gb_at_144=56.0):
    """N > 1 runs one box of n^3 trilinear hexahedra per rank; the setup of a 144^3 box peaks at 52 GB of host memory per
    rank (profiles/r02_bench_n4_configs4.json).  When world x 56 GB does not fit into 85 % of the node's memory the box
    is shrunk in steps of 16 (5 levels need a multiple of 16) -- a guard against driving the node out of memory, stated in
    config.workload when it fires."""
    mem = host_memory_gb()
    if world <= 1 or mem <= 0.0:
        return n
    while n > 48 and world * per_rank_gb_at_144 * (n / 144.0) ** 3 > 0.85 * mem:
        n -= 16
    return n


def product_level_operators(ctx, ns, lv, deformed=False):
    """Level operators (A0, [P_l], [D_l]) of the bounded CPU sample, taken from the PRODUCT's hierarchy of the same
    workload (inputs of the solve path; what is timed on the CPU is the oracle V-cycle over them).  deformed: one box
    of the configs[4] geometry (the unit cube after the 3DHdivWeakScaling vertex map, essential attributes 2-5)."""
    import scipy.sparse as sp
    from parelag_b200 import api
    if deformed:
        X = api.box_vertex_coords((1, 1, 1), (0, 0, 0), (ns, ns, ns), api.weak_scaling_deformation)
        Ss = api.Sequence.hex((ns, ns, ns), lv, jstart=1, coords=X)
        ess = np.array([0, 1, 1, 1, 1, 0], dtype=np.int32)
    else:
        Ss = api.Sequence.hex((ns, ns, ns), lv, jstart=1)
        ess = ESS
    As = Ss.assemble_system(ctx, 0, 2, ess).to_scipy()
    bit = sum(1 << a for a in range(6) if ess[a])
    Ps, Ds = [], []
    for l in range(lv):
        D = Ss.get_csr(l, "D", 1)
        m = (Ss.get_bdr_mask(l, 1) & bit) != 0
        Ds.append(sp.csr_matrix((np.where(m[D.indices], 0.0, D.data), D.indices, D.indptr), shape=D.shape))
        if l + 1 < lv:
            P = Ss.get_csr(l, "P", 2)
            mc = (Ss.get_bdr_mask(l + 1, 2) & bit) != 0
            Ps.append(sp.csr_matrix((np.where(mc[P.indices], 0.0, P.data), P.indices, P.indptr), shape=P.shape))
    Ss.free()
    return As, Ps, Ds


def workload_name(gpus, n, ndofs_box, levels, deformed):
    """the part of config.workload both arms share"""
    if deformed:
        return ("3DHdivWeakScaling (configs[4]): one box of %d^3 trilinear hexahedra per GPU (unit cube after y += exp(z)/2, "
                "x += sin(y), essential attributes 2-5), H(div) A=M2+D2^T M3 D2, %d-level AMGe, Hiptmair(l1-GS,l1-GS), "
                "PCG-GS coarse solver" % (n, levels))
    return ("MultigridTest2Form (configs[1]): H(div) A=M2+D2^T M3 D2, %d^3 hexahedra, %d RT0 dofs, %d-level AMGe, "
            "Hiptmair(l1-GS,l1-GS), PCG-GS coarse solver" % (n, ndofs_box, levels))


MIXED_SOLVER_NAME = {"ldu": "Block LDU with AMGe V-cycles (l1-GS) on M (Forms 2) and on the DIAGONAL Schur complement (Forms 3); step = one "
                            "preconditioner application (3 + 1 V-cycles)",
                     "blocked": "blocked AMGe (Forms 2 3) with a Block Jacobi smoother (l1-GS on M and on the Schur complement); step = one "
                                "blocked V-cycle"}


def other_workload_name(cfg, n, ndofs, levels, args):
    if cfg == "cfg1":
        return ("MultigridTest0Form (configs[0]): H1 Laplacian A=D0^T M1 D0 on meshes/cube456.mesh refined %d times (tetrahedra), "
                "%d dofs, %d-level AMGe by derefinement, l1-GS smoothers, PCG-GS coarse solver" % (args.nref, ndofs, levels))
    if cfg == "hcurl":
        return ("MultigridTest1Form (configs[2]): H(curl) A=M1+D1^T M2 D1, %d^3 hexahedra, %d Nedelec dofs, %d-level AMGe, "
                "Hiptmair(l1-GS,l1-GS) with the H1 auxiliary space, PCG-GS coarse solver" % (n, ndofs, levels))
    if cfg == "darcy":
        return ("MultigridTestDarcy (configs[1]): mixed system [[M B^T][B 0]], %d^3 hexahedra, %d dofs (RT0 + L2), %d levels, GMRES(50) + %s"
                % (n, ndofs, levels, MIXED_SOLVER_NAME[args.mixed_solver]))
    if getattr(args, "perm_file", None):
        return ("MultigridTestSPE10 (configs[3]): 60x220x85 cells of 20x10x2, SPE10 permeability tensor from %s, mixed system "
                "[[M B^T][B 0]], %d dofs, %d levels (logical Cartesian agglomeration with ragged blocks), GMRES(50) + %s"
                % (os.path.basename(args.perm_file), ndofs, levels, MIXED_SOLVER_NAME[args.mixed_solver]))
    return ("MultigridTestSPE10-shaped (configs[3]): 60x220x85 cells of 20x10x2, synthetic lognormal permeability (4+ decades), mixed "
            "system [[M B^T][B 0]], %d dofs, %d levels (logical Cartesian agglomeration with ragged blocks), GMRES(50) + %s"
            % (ndofs, levels, MIXED_SOLVER_NAME[args.mixed_solver]))


def levels_for(n, cap):
    lv = 1
    while n % (2 ** lv) == 0 and lv < cap:
        lv += 1
    return lv


def cpu_setup_baseline(n=16, levels=4):
    """Setup half of the metric on the CPU: the oracle's Coarsen() of all levels (oracle/amge.py: numpy + LAPACK
    restatement of DeRhamSequence::Coarsen, one thread, Python loops over the agglomerates) on a bounded sample."""
    from oracle import amge
    t0 = time.perf_counter()
    mesh, seqs = amge.build_hierarchy((n, n, n), levels, jstart=1)
    t = time.perf_counter() - t0
    nd = int(seqs[0].dof[2].ndofs)
    return {"seconds": t, "sample": "oracle Coarsen() of %d levels on %d^3 hexahedra (%d RT0 dofs), forms 1-3" % (levels, n, nd),
            "dofs_per_s": nd / t, "cores": 1, "kind": "port (numpy restatement, Python loops: an upper bound on the CPU time, "
            "not a tuned C++ build)", "seconds_scaled_to_9020160_dofs": t * 9020160.0 / nd}


def run_reference(args, rank):
    """CPU arm: the oracle's V-cycle (hypre/MFEM arithmetic restated in C, oracle/solve_oracle.c) with all the host
    threads this process may use -- one row block per thread = one MPI rank per core, hybrid Gauss-Seidel -- on a
    bounded sample of the N = 1 workload (same operator, smoother, coarse solver; ref_n^3 instead of 144^3 hexahedra).
    Level operators come from the product's hierarchy when a GPU is present (inputs only), else from the oracle's."""
    if rank != 0:
        return
    cores = host_threads()
    os.environ["OMP_NUM_THREADS"] = str(cores)          # a launcher (torchrun) exports OMP_NUM_THREADS=1
    os.environ.pop("OMP_THREAD_LIMIT", None)
    from oracle import solve as orc
    got = orc.set_threads(cores)
    assert got == cores, "OpenMP gives %d threads, %d requested" % (got, cores)
    deformed = args.gpus > 1 and not args.no_deform     # the N > 1 arm runs configs[4]: sample = ONE box of it
    n_s = args.ref_n
    if n_s <= 0 and fit_box_size(args.n, args.gpus) != args.n:
        n_s = fit_box_size(args.n, args.gpus)            # the box size the GPU arm takes on this node (memory guard)
    if n_s <= 0:
        # the full per-GPU size when the host has the memory for the oracle's copies of the hierarchy (~60 GB at 144^3)
        avail = 0
        try:
            avail = int([l for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0].split()[1]) >> 20
        except Exception:
            pass
        n_s = args.n if avail >= 120 else 96
    inputs, src = oracle_hierarchy_inputs, "oracle"
    try:
        import torch
        if torch.cuda.is_available():
            from parelag_b200 import api
            ctx = api.session(rank=0, nranks=1, device=0)
            inputs, src = (lambda ns, lv: product_level_operators(ctx, ns, lv, deformed)), "product"
    except Exception:
        pass
    if src == "oracle":
        n_s, deformed = min(n_s, 32), False              # the numpy coarsening oracle: minutes beyond that
    levels = levels_for(n_s, args.levels)
    H, ndofs = cpu_vcycle_setup(n_s, levels, cores, inputs)
    t, done, z = time_cpu_vcycles(H, ndofs, args.steps, min(args.warmup, 1), budget_s=120.0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"z": z})
    value = ndofs / t
    setup = None if args.no_cpu_setup else cpu_setup_baseline()
    sample = ("H(div) AMGe V-cycle (Hiptmair l1-GS, PCG-GS coarse) on %d^3 hexahedra, %d RT0 dofs, %d levels (level operators "
              "from the %s); SpMV and hybrid GS with %d OpenMP threads = %d row blocks (one MPI rank per core), oracle "
              "port of the hypre/MFEM kernels" % (n_s, ndofs, levels, src, cores, cores))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": done, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * t, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.gpus, n_s, ndofs, levels, deformed),
                       "sample": "one box (%d^3 hexahedra, %d RT0 dofs) of the workload, %d host threads" % (n_s, ndofs, cores),
                       "gs_order": "natural within a row block, one row block per thread (hypre's hybrid scheme)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "omp_threads": got, "kind": "port", "sample": sample,
                             "setup": setup},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)
    sys.stdout.flush()
    os._exit(0)


# ----------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", "--n", dest="n", type=int, default=144, help="hexahedra per direction (144 -> 9.02M RT0 dofs)")
    ap.add_argument("--levels", type=int, default=5)
    ap.add_argument("--ordering", default="multicolor", choices=["multicolor", "natural"])
    ap.add_argument("--jstart", type=int, default=0, help="jformStart of the sequence (driver uses 0)")
    ap.add_argument("--ref-n", type=int, default=0,
                    help="hexahedra per direction of the CPU arm's sample (0: --size if the host has >= 120 GB free, else 96)")
    ap.add_argument("--no-cpu-setup", action="store_true", help="skip the CPU setup baseline (oracle Coarsen on 16^3)")
    ap.add_argument("--no-deform", action="store_true", help="N > 1: axis-aligned boxes instead of the configs[4] geometry")
    ap.add_argument("--deform", action="store_true",
                    help="N = 1: run ONE box of the configs[4] workload (trilinear hexahedra, essential attributes 2-5) instead of "
                         "configs[1] -- the like-for-like base of the N > 1 weak-scaling lines")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity block")
    ap.add_argument("--no-weak-base", action="store_true",
                    help="N = 1: skip the extra leg that times one box of configs[4] (the base of the N > 1 weak-scaling lines)")
    ap.add_argument("--config", default="hdiv", choices=["hdiv", "cfg1", "hcurl", "darcy", "spe10"],
                    help="N = 1 workload: hdiv = BASELINE configs[1] MultigridTest2Form (the headline), cfg1 = configs[0] "
                         "MultigridTest0Form (H1 on meshes/cube456.mesh, --nref refinements, 3 levels), hcurl = configs[2] "
                         "MultigridTest1Form (--size 192), darcy = configs[1] MultigridTestDarcy (--size 136, 4 levels), "
                         "spe10 = configs[3] (60x220x85 cells, synthetic lognormal permeability, mixed Darcy)")
    ap.add_argument("--mixed-solver", default="ldu", choices=["ldu", "blocked"],
                    help="darcy / spe10: GMRES + Block LDU with AMGe V-cycles on M and on the Schur complement (spe10_example_parameters.xml; a "
                         "step = one application of that preconditioner), or GMRES + the blocked AMGe hierarchy with a Block Jacobi "
                         "smoother (darcy_example_parameters.xml; a step = one blocked V-cycle)")
    ap.add_argument("--nref", type=int, default=4, help="cfg1: uniform refinements of cube456.mesh (driver: 2 serial + 2 parallel)")
    ap.add_argument("--cpu-n", type=int, default=32, help="bounded sample of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sell-min-rows", type=int, default=None,
                    help="tuning: levels with fewer rows use the lanes-per-row CSR Gauss-Seidel kernel (library default 200000)")
    ap.add_argument("--gs-slabs", type=int, default=None, help="tuning: PE_TUNE_GS_SLABS (slab-major multicolour order on >= 4M-row levels)")
    ap.add_argument("--fused-gs-mb", type=int, default=None, help="tuning: PE_TUNE_FUSED_GS_MAX_MB (0 = one launch per colour)")
    ap.add_argument("--perm-file", default=None,
                    help="--config spe10: path of the SPE10 permeability file (spe_perm.dat); default: synthetic lognormal field")
    ap.add_argument("--halo", default="p2p", choices=["p2p", "nccl"],
                    help="multi-GPU halo exchange: NVLink peer-memory stores (default) or ncclSend/ncclRecv")
    ap.add_argument("--profile-range", action="store_true",
                    help="bracket 2 extra V-cycles with cudaProfilerStart/Stop (ncu --profile-from-start off) and exit")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (the preconditioned vector z; z_rank<r> per "
                         "rank when N > 1) as DIR/<name>.npy in float64, at most 64 MB in all: a longer vector is stored at a "
                         "fixed, seeded sample of its entries.  The inputs depend on the arguments only, so two builds can be "
                         "compared file by file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    args.warmup = max(args.warmup, 3)
    # host threads of the setup (OpenMP in the host integer work): torchrun exports OMP_NUM_THREADS=1, which made the
    # multi-rank setup single-threaded; every rank gets its share of the cores instead (set before libgomp is loaded)
    os.environ["OMP_NUM_THREADS"] = str(max(1, host_threads() // max(world, 1)))

    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl")

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(v):
        if dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    from parelag_b200 import api, capi
    n, levels = args.n, args.levels
    if world > 1 and args.config == "hdiv":
        fit = fit_box_size(n, world)                     # from MemTotal / the cgroup limit: the same on every rank of the node
        if fit != n and rank == 0:
            print("bench.py: %d ranks x %d^3 boxes do not fit the node's %.0f GB of host memory; running %d^3 boxes"
                  % (world, n, host_memory_gb(), fit), file=sys.stderr, flush=True)
        n = fit
    procs = {1: (1, 1, 1), 2: (2, 1, 1), 4: (2, 2, 1), 8: (2, 2, 2)}.get(world)
    if procs is None:
        raise SystemExit("bench.py: --gpus must be 1, 2, 4 or 8")
    capi.set_tuning(capi.TUNE_P2P_HALO, 1 if args.halo == "p2p" else 0)
    if world > 1:
        # one box per GPU: the library's own NCCL communicator carries the data path, a gloo group the
        # setup-time host exchanges (MPI in the reference)
        from parelag_b200 import par
        ids = [capi.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        ctx = api.session(rank=rank, nranks=world, device=local_rank, nccl_id=ids[0])
        api.set_host_comm(par.HostComm(dist.new_group(backend="gloo")))
    else:
        ctx = api.session(rank=0, nranks=1, device=local_rank)
    api.lib().pe_api_timer_clear()
    if args.sell_min_rows is not None:
        capi.set_tuning(capi.TUNE_SELL_MIN_ROWS, args.sell_min_rows)
    if args.gs_slabs is not None:
        capi.set_tuning(capi.TUNE_GS_SLABS, args.gs_slabs)
    if args.fused_gs_mb is not None:
        capi.set_tuning(capi.TUNE_FUSED_GS_MAX_MB, args.fused_gs_mb)

    cfg = args.config
    if world > 1 and cfg != "hdiv":
        raise SystemExit("bench.py: --config %s is a single-GPU workload" % cfg)
    mixed = cfg in ("darcy", "spe10")
    form = {"hdiv": 2, "hcurl": 1, "cfg1": 0}.get(cfg, 2)
    if cfg == "hcurl" and args.n == 144:
        n, levels = 192, 4
    if cfg == "darcy" and args.n == 144:
        n, levels = 136, 4
    if cfg == "spe10":
        levels = 4
    # ---------------- parity block (the oracle is the checker; nothing of it is timed or shipped)
    deformed = (world > 1 and not args.no_deform) or (world == 1 and args.deform and cfg == "hdiv")
    ess = np.array([0, 1, 1, 1, 1, 0], dtype=np.int32) if deformed else ESS     # 3DHdivWeakScaling.cpp:53-66
    parity = None
    host_group = api._host_comm.group if world > 1 else None
    if not args.no_parity and cfg == "hdiv":
        try:
            from tests import parity_checks
            if world > 1:
                parity = dict(parity_checks.multi_rank(ctx, rank, world, deform=deformed, group=host_group), ok=True)
            else:
                parity = dict(parity_checks.single_rank_small(ctx), ok=True)
        except AssertionError as e:
            parity = {"ok": False, "failed": repr(e)[:400]}
        if world > 1:
            oks = [None] * world
            dist.all_gather_object(oks, bool(parity["ok"]), group=host_group)
            parity["ok"] = bool(all(oks))
        api.lib().pe_api_timer_clear()

    # ---------------- setup (timed with the reference's timer names)
    t0 = time.perf_counter()
    if deformed and world == 1:
        X = api.box_vertex_coords(procs, (0, 0, 0), (n, n, n), api.weak_scaling_deformation)
        S = api.Sequence.hex((n, n, n), levels, jstart=max(args.jstart, 1), coords=X)
        del X
    elif deformed:
        X = api.box_vertex_coords(procs, api.rank_box(procs, rank), (n, n, n), api.weak_scaling_deformation)
        S = api.Sequence.hex_par(procs, (n, n, n), levels, jstart=max(args.jstart, 1), coords=X)
        del X
    elif world > 1:
        S = api.Sequence.hex_par(procs, (n, n, n), levels, L=(1.0, 1.0, 1.0), jstart=args.jstart)
    elif cfg == "cfg1":
        levels = 3
        msh = np.load(os.path.join(ROOT, "tests", "golden", "cube456.npz"))      # arrays of meshes/cube456.mesh (tests/golden/make_cube456.py)
        S = api.Sequence.tet(msh["vertices"], msh["tets"], msh["bdr_triangles"], msh["bdr_attributes"], args.nref, levels, jstart=0)
    elif cfg == "hcurl":
        S = api.Sequence.hex((n, n, n), levels, jstart=0)
    elif cfg == "darcy":
        S = api.Sequence.hex((n, n, n), levels, jstart=2)
    elif cfg == "spe10":
        # SPE10-shaped (InversePermeabilityFunction.cpp:254-259: 60 x 220 x 85 cells of 20 x 10 x 2 ft); synthetic
        # lognormal permeability (the data set is not available offline): log10 k ~ N(-1, 1.5^2) clipped to [-4, 2]
        dims, Lspe = (60, 220, 85), (1200.0, 2200.0, 170.0)
        if args.perm_file:
            # the real data set when the user has it (data/spe_perm.dat, examples/MultigridTestSPE10.cpp:85,181-183): read
            # and evaluated as the reference does, diagonal tensor coefficient (1/K_x, 1/K_y, 1/K_z) per cell
            api.spe10_read(args.perm_file, dims, (20.0, 10.0, 2.0))
            S = api.Sequence.spe10(dims, (20.0, 10.0, 2.0), levels, jstart=2)
        else:
            kinv = 10.0 ** (-np.clip(np.random.default_rng(13).normal(-1.0, 1.5, size=dims[0] * dims[1] * dims[2]), -4.0, 2.0))
            S = api.Sequence.hex(dims, levels, L=Lspe, beta=kinv, jstart=2)
    else:
        S = api.Sequence.hex((n, n, n), levels, jstart=args.jstart)
    ctx.sync()
    t_coarsen = time.perf_counter() - t0
    import ctypes
    st6 = (ctypes.c_double * 6)()
    capi.lib().pe_local_stage_seconds(st6, 1)
    ext_stages = {"h2d_s": st6[0], "kernel_s": st6[1], "d2h_s": st6[2], "h2d_GB": st6[3] / 1e9, "d2h_GB": st6[4] / 1e9,
                  "calls": int(st6[5])}
    t0 = time.perf_counter()
    blocks = None
    if mixed:
        Mb, Bb, Btb = S.assemble_darcy(ctx, 0)
        blocks = [[Mb, Btb], [Bb, None]]
        A = Mb                                # the SpMV figure is taken on the H(div) mass block
        ndofs = Mb.info()[0] + Bb.info()[0]
    else:
        A = S.assemble_system(ctx, 0, form, ess)
        ndofs = A.info()[0]                   # true dofs owned by this rank
    ctx.sync()
    t_assemble = time.perf_counter() - t0
    nrows0 = A.info()[0]
    nnz0 = A.info()[3] + A.info()[4]

    def sum_over_ranks(v):
        if dist is None:
            return v
        t = torch.tensor([float(v)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())
    ndofs_global = int(round(sum_over_ranks(ndofs)))
    peak, peak_src = peaks()
    # ---------------- SpMV alone on the fine operator (the "SpMV HBM GB/s vs peak" part of the metric)
    A2 = A
    xs, ys = capi.Vec(ctx, data=np.random.default_rng(99 + rank).standard_normal(nrows0)), capi.Vec(ctx, nrows0)
    for _ in range(3):
        A2.spmv(xs, ys)
    ctx.sync(); ctx.timer_start()
    for _ in range(20):
        A2.spmv(xs, ys)
    ms_spmv = ctx.timer_stop() / 20
    b_spmv = 12.0 * nnz0 + 4.0 * (nrows0 + 1) + 16.0 * nrows0
    spmv = {"ms": ms_spmv, "GBs": b_spmv / ms_spmv / 1e6, "frac_of_measured_peak": b_spmv / ms_spmv / 1e6 / peak,
            "nnz": nnz0, "rows": nrows0}

    # full-size kernel parity (N = 1): one SpMV and one multicolour GS sweep of THIS operator against solve_oracle.c
    if parity is not None and parity.get("ok") and world == 1 and cfg == "hdiv" and not args.profile_range:
        try:
            parity["full_size"] = parity_checks.full_size_kernels(ctx, A)
        except AssertionError as e:
            parity["ok"] = False
            parity["failed"] = repr(e)[:400]
    t0 = time.perf_counter()
    if mixed and args.mixed_solver == "ldu":
        solver = api.BlockSolver(api.library_xml(library_darcy_ldu(args.ordering)), "GMRES with Block LDU", blocks, S, 0, [2, 3],
                                 ess_attr=np.zeros((2, 6), dtype=np.int32))
    elif mixed:
        solver = api.BlockSolver(api.library_xml(library_darcy(args.ordering)), "GMRES with blocked AMGe", blocks, S, 0, [2, 3])
    elif cfg == "cfg1":
        solver = api.Solver(api.library_xml(library_h1(args.ordering)), "PCG with Auxiliary Space Preconditioner", A, S, 0, 0, ess)
    else:
        solver = api.Solver(api.library_xml(library(args.ordering, form)), "PCG with Auxiliary Space Preconditioner",
                            A, S, 0, form, ess)
    ctx.sync()
    t_build = time.perf_counter() - t0
    try:
        nlev = solver.num_levels()
        level_info = [solver.level_info(l) for l in range(nlev)]
    except Exception:                         # blocked hierarchy: the level operators are block operators
        nlev, level_info = levels, []
    # the reference's TimeManager names (examples/MultigridTest2Form.cpp:248-375, AMGeSolverFactory.cpp)
    timers = {}
    for l in range(levels):
        for nm in ("Mesh Agglomeration -- Level %d" % l, "DeRhamSequence Construction -- Level %d" % l,
                   "Build smoother: level %d" % l, "Build coarse solver: level %d" % l):
            v = api.timer(nm)
            if v > 0:
                timers[nm] = v
    for nm in ("Build Hierarchy: build from deRham Sequence", "SharingMap construction", "Assemble linear system",
               "Coarsen: DofAgglomeration", "Coarsen: traces prepare (host)", "Coarsen: batched traces (H2D + kernels + D2H)",
               "Coarsen: traces commit (host)", "Coarsen: extension prepare (host)",
               "Coarsen: batched extension (H2D + kernels + D2H)", "Coarsen: extension commit (host)",
               "Coarsen: finalize P and D", "Coarsen: project targets", "Host arena reserve (parallel first touch)",
               "Fine sequence: dof handlers", "Fine sequence: D and mass pools", "Fine sequence: targets"):
        v = api.timer(nm)
        if v > 0:
            timers[nm] = v

    # ---------------- device-resident V-cycle steps
    rng = np.random.default_rng(1234 + rank)
    r_host = rng.standard_normal(ndofs)
    r_dev, z_dev = capi.Vec(ctx, data=r_host), capi.Vec(ctx, ndofs)
    for _ in range(args.warmup):
        solver.prec_mult_device(r_dev, z_dev)
    ctx.sync()
    if args.profile_range:
        rt = torch.cuda.cudart()
        rt.cudaProfilerStart()
        for _ in range(2):
            solver.prec_mult_device(r_dev, z_dev)
        ctx.sync()
        rt.cudaProfilerStop()
        print(json.dumps({"profile_range": "2 V-cycles", "ndofs": int(ndofs)}))
        return
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    l0 = ctx.launch_count()
    ctx.sync()
    ctx.timer_start()
    for _ in range(args.steps):
        solver.prec_mult_device(r_dev, z_dev)
    ms = ctx.timer_stop()
    barrier()
    launches = ctx.launch_count() - l0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"z" if world == 1 else "z_rank%d" % rank: z_dev.download()}, DUMP_MAX_BYTES // world)
    ms = max_over_ranks(ms)
    ms_per_step = ms / args.steps
    value = ndofs_global / (ms_per_step * 1e-3)

    # ---------------- roofline of the dominant kernel
    peak, peak_src = peaks()
    OPN = {1: "sell_spmv", 2: "sell_gs", 3: "csr_spmv", 4: "perm_in", 5: "perm_out", 6: "axpby", 7: "add3", 8: "fill",
           9: "copy", 10: "scale", 11: "mul", 12: "dot", 13: "dot_fin", 14: "axpy_dev", 15: "xpby_dev", 16: "pcg_step"}
    try:
        prog = solver.program()
    except Exception:                         # the preconditioner is not a Hierarchy (Block LDU of the mixed configs)
        prog = None
    if prog is not None:
        # the whole V-cycle is ONE persistent kernel (k_program): its launch duration is the step;
        # algorithmic bytes = sum over the recorded ops (DESIGN.md section 4; permutation ops count 0)
        nops, pbytes = prog
        achieved = pbytes / (ms_per_step * 1e-3) / 1e9
        t_op, us_op, by_op = solver.program_profile(ctx)
        ops = {}
        for k in sorted(set(t_op.tolist())):
            m = t_op == k
            ops[OPN.get(k, str(k))] = {"count": int(m.sum()), "us": float(us_op[m].sum()),
                                       "GBs": float(by_op[m].sum() / max(us_op[m].sum(), 1e-9) / 1e3)}
        big = by_op > 64e6      # fine-level ops: individually HBM-bound
        roofline = {"bound": "hbm", "kernel": "k_program (whole V-cycle, %d ops, 1 launch per step)" % nops,
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "frac_of_8TBs_spec": achieved / 8000.0, "peak_source": peak_src, "launches": args.steps,
                    "avg_launch_us": 1e3 * ms_per_step, "algorithmic_bytes_per_launch": pbytes,
                    "traffic": traffic_from_profiles().get("k_program"), "share_of_step": 1.0,
                    "profiled_launch_us": float(us_op.sum()),
                    "fine_level_ops": {"count": int(big.sum()), "us": float(us_op[big].sum()),
                                       "GBs": float(by_op[big].sum() / max(us_op[big].sum(), 1e-9) / 1e3)},
                    "ops": ops}
    else:
        # kernel-by-kernel path: separate profiled pass over the same steps
        ctx.profile(True)
        for _ in range(args.steps):
            solver.prec_mult_device(r_dev, z_dev)
        ctx.profile(False)
        names = {0: "k_sell_spmv", 1: "k_sell_gs (fine-level colour launches, >= 64 MB each)", 2: "k_jacobi_update",
                 3: "k_gs_set / small k_sell_gs (coarse levels)"}
        prof = {names[i]: ctx.profile_get(i) for i in names}
        dom = max(prof, key=lambda k: prof[k][1])
        cnt, pms, pbytes = prof[dom]
        achieved = pbytes / (pms * 1e-3) / 1e9 if pms > 0 else 0.0
        tr = traffic_from_profiles().get(dom.split(" ")[0])
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "frac_of_8TBs_spec": achieved / 8000.0, "peak_source": peak_src,
                    "launches": cnt, "avg_launch_us": 1e3 * pms / max(cnt, 1),
                    "algorithmic_bytes_per_launch": pbytes / max(cnt, 1), "traffic": tr,
                    # share of the kernel time of the kernel-by-kernel pass (every launch bracketed by events, like
                    # the serialised ncu launch list it is compared with); the graph replay of the timed region
                    # has no per-kernel clock
                    "share_of_step": pms / max(sum(v[1] for v in prof.values()), 1e-9),
                    "share_basis": "event-bracketed kernel-by-kernel pass over the same steps (SpMV + GS + Jacobi kernels)",
                    "all": {k: {"launches": v[0], "ms": v[1], "GBs": (v[2] / (v[1] * 1e-3) / 1e9 if v[1] > 0 else 0.0)}
                            for k, v in prof.items()}}

    # ---------------- end to end through the plugin API with pinned HOST buffers
    b_pin = torch.empty(ndofs, dtype=torch.float64).pin_memory()
    x_pin = torch.empty(ndofs, dtype=torch.float64).pin_memory()
    b_np, x_np = b_pin.numpy(), x_pin.numpy()
    b_np[:] = r_host
    # the reference-facing call: mfem::Solver::Mult(B, X) of the AMGe Hierarchy with HOST vectors
    # (pe_api_solver_prec_mult: H2D of b from pinned memory, V-cycle, D2H of x, all inside the call)
    for _ in range(2):
        solver.prec_mult_into(b_np, x_np)
    barrier()
    ctx.sync()
    ctx.timer_start()
    for _ in range(args.steps):
        solver.prec_mult_into(b_np, x_np)
    ms_e2e = max_over_ranks(ctx.timer_stop()) / args.steps
    e2e = {"value": ndofs_global / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
           "call": "pe_api_solver_prec_mult (Hierarchy::Mult with pinned host vectors)",
           "h2d_bytes_per_step": 8 * ndofs_global, "d2h_bytes_per_step": 8 * ndofs_global}

    # ---------------- one full PCG solve (iterations, residual history) through host buffers
    bvec = rng.standard_normal(ndofs)
    t0 = time.perf_counter()
    x = solver.mult(bvec)
    t_solve = time.perf_counter() - t0
    hist, iters, conv = solver.history()

    # ---------------- like-for-like base of the N > 1 weak-scaling lines: ONE box of configs[4] on this GPU
    weak_base = None
    if world == 1 and cfg == "hdiv" and not deformed and not args.no_weak_base and not args.profile_range:
        try:
            solver.free(); S.free()
            t0 = time.perf_counter()
            Xd = api.box_vertex_coords((1, 1, 1), (0, 0, 0), (n, n, n), api.weak_scaling_deformation)
            Sd = api.Sequence.hex((n, n, n), levels, jstart=1, coords=Xd)
            del Xd
            essd = np.array([0, 1, 1, 1, 1, 0], dtype=np.int32)
            Ad = Sd.assemble_system(ctx, 0, 2, essd)
            nd = Ad.info()[0]
            sd = api.Solver(api.library_xml(library(args.ordering)), "PCG with Auxiliary Space Preconditioner", Ad, Sd, 0, 2, essd)
            ctx.sync()
            t_setup_d = time.perf_counter() - t0
            rd, zd = capi.Vec(ctx, data=rng.standard_normal(nd)), capi.Vec(ctx, nd)
            for _ in range(3):
                sd.prec_mult_device(rd, zd)
            ctx.sync(); ctx.timer_start()
            for _ in range(10):
                sd.prec_mult_device(rd, zd)
            ms_d = ctx.timer_stop() / 10
            sd.mult(rng.standard_normal(nd))
            _, it_d, conv_d = sd.history()
            weak_base = {"workload": workload_name(1, n, nd, sd.num_levels(), True), "ms_per_step": ms_d, "value": nd / (ms_d * 1e-3),
                         "unit": UNIT, "steps": 10, "setup_s": t_setup_d, "pcg_iterations": it_d, "pcg_converged": conv_d,
                         "levels": [{"rows": li[0], "nnz": li[1]} for li in (sd.level_info(l) for l in range(sd.num_levels()))],
                         "note": "the N > 1 lines run this box per GPU: weak-scaling efficiency = value_N / (N x this value)"}
            sd.free(); Sd.free()
        except Exception as e:                    # the headline line must not depend on this leg
            weak_base = {"failed": repr(e)[:300]}

    line = None
    if rank == 0:
        cpu_baseline = None
        if not args.no_cpu_baseline and world == 1 and cfg == "hdiv":
            from oracle import solve as orc
            orc.set_threads(1)
            lv = levels_for(args.cpu_n, levels)
            H, nd = cpu_vcycle_setup(args.cpu_n, lv, 1, lambda ns, lvv: product_level_operators(ctx, ns, lvv))
            t_cpu, done, _ = time_cpu_vcycles(H, nd, 30, 1, budget_s=20.0)
            cpu_baseline = {"value": nd / t_cpu, "unit": UNIT, "cores": 1, "kind": "port",
                            "sample": "same H(div) AMGe V-cycle (Hiptmair l1-GS natural order, PCG-GS coarse) on a "
                                      "%d^3-hexahedra sample (%d RT0 dofs, %d levels), %d cycles of %.3f s on one host core; "
                                      "oracle port of the hypre/MFEM kernels (oracle/solve_oracle.c)"
                                      % (args.cpu_n, nd, lv, done, t_cpu),
                            "setup": None if args.no_cpu_setup else cpu_setup_baseline()}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": other_workload_name(cfg, n, ndofs, nlev, args) if cfg != "hdiv" else
                                       workload_name(world, n, ndofs, nlev, deformed) if (world == 1 or deformed) else
                                       ("3DHdivWeakScaling layout, axis-aligned: %dx%dx%d boxes of %d^3 hexahedra, one box per GPU, all "
                                        "attributes essential, H(div) A=M2+D2^T M3 D2, %d-level AMGe, Hiptmair(l1-GS,l1-GS), PCG-GS "
                                        "coarse solver" % (procs + (n, nlev))),
                           "boxes": "%dx%dx%d" % procs, "global_true_dofs": ndofs_global,
                           "scaling_note": ("N = 1 runs configs[1] (axis-aligned cube); N > 1 runs configs[4] (trilinear hexahedra: the "
                                            "coarse spaces carry NullSpace dofs, 2.3x the rows and 5x the non-zeros on level 1, ~2.5x the "
                                            "V-cycle work per fine dof).  The like-for-like weak-scaling base of the N > 1 lines is "
                                            "`bench.py --gpus 1 --deform` (profiles/), not the N = 1 headline line."),
                           "gs_order": "%s within a rank, frozen ghosts across ranks (hypre's hybrid scheme)" % args.ordering,
                           "halo": (None if world == 1 else
                                    "NVLink peer-memory stores + device flags (CUDA IPC)" if capi.lib().pe_ctx_p2p_enabled(ctx.h)
                                    else "NCCL send/recv"),
                           "l2_policy": "inputs larger than L2 (hierarchy working set %.1f GB)" %
                                        (sum(12.0 * li[1] for li in level_info) / 1e9),
                           "parallelism": ("single GPU" if world == 1 else
                                           "domain decomposition, %d ranks = %d GPUs, one mesh box each" % (world, world)),
                           "jform_start": args.jstart,
                           "tuning": {"sell_min_rows": capi.get_tuning(capi.TUNE_SELL_MIN_ROWS), "gs_slabs": capi.get_tuning(capi.TUNE_GS_SLABS),
                                      "fused_gs_max_mb": capi.get_tuning(capi.TUNE_FUSED_GS_MAX_MB), "pdl": capi.get_tuning(capi.TUNE_PDL)},
                           "levels": [{"rows": li[0], "nnz": li[1], "nnz_P": li[2]} for li in level_info]},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "parity": parity, "weak_scaling_base": weak_base,
                "roofline": roofline, "cpu_baseline": cpu_baseline,
                "setup_s": {"sequence_all_levels": t_coarsen, "assemble_system": t_assemble, "build_solver": t_build,
                            "total": t_coarsen + t_assemble + t_build, "timers": timers,
                            "batched_extension_stages": ext_stages,
                            "host_peak_rss_GB": __import__("resource").getrusage(__import__("resource").RUSAGE_SELF).ru_maxrss / 1e6,
                            "host_cores": os.cpu_count()},
                "spmv_fine_operator": spmv,
                "pcg": {"iterations": iters, "converged": conv, "seconds_host_buffers": t_solve,
                        "Br_r_first": float(hist[0]), "Br_r_last": float(hist[-1])}}
        print(json.dumps(line), flush=True)
    if dist is not None:
        # leave without running interpreter teardown: destroying torch's NCCL group while this library's
        # own communicator still owns captured graphs was observed to hang at exit
        dist.barrier()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
