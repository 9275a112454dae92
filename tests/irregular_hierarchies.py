"""Irregular AMGe hierarchies of the oracle and the SELL kernel variants they reach (tests/test_vcycle_irregular_gpu.py,
tests/test_irregular_variants_cpu.py).

Hierarchies, all built by the oracle on the CPU:
  - deformed:     16^3 hexahedra under the configs[4] map (amge.weak_scaling_deformation), 4 levels, forms 0-2,
                  essential attributes [0,1,1,1,1,0] as bench.py sets them for the deformed geometry;
  - tets:         cube456 (configs[0]) refined twice, 3 levels, form 0;
  - coefficients: uniform 16^3, 4 levels, forms 1 and 2, lognormal alpha and beta over four decades.

Predictor of the entry-group variant (pe_sell.cu sell_pick_group) of every k_sell_gs / k_sell_spmv launch, with the
rules of the host code:
  - a multicolour SELL sweep stores the rows colour by colour (the oracle's greedy colouring, rows of one colour in
    ascending order), each colour padded to whole slices of 32 rows; a slice is as wide as its longest row and a colour
    launch takes the group of its widest slice;
  - G = PE_TUNE_SELL_GROUP when that is 4, 8 or 12, else 4 / 8 / 12 / 8 / 4 for widths <= 4 / <= 8 / <= 12 / <= 24 /
    larger; single-group when the widest slice fits one group;
  - one sweep is a forward pass over the colours and a backward pass; from a zero initial guess the first non-empty
    colour of the forward pass is done by the renumbering pass (no k_sell_gs launch), and the backward pass skips the
    last colour when every row of that colour has l1 norm == diagonal > 0 (l1-Gauss-Seidel, unit weights, one rank);
  - one count is 32 padded slice rows per slice of the launch.
"""
import os

import numpy as np

from oracle import amge, drivers, solve as orc, tets

MESH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cube456.npz")
ESS_ALL = np.ones(6, dtype=np.int32)
ESS_DEFORMED = np.array([0, 1, 1, 1, 1, 0], dtype=np.int32)      # bench.py, 3DHdivWeakScaling.cpp:53-66
GROUPS = (4, 8, 12)
CHOICES = [(G, single) for G in GROUPS for single in (True, False)]


# ---------------------------------------------------------------------------------------------------------------------
# hierarchies
# ---------------------------------------------------------------------------------------------------------------------
def lognormal(n, seed):
    """lognormal coefficients over four decades: 10^x, x ~ N(0, 0.7) clipped to [-2, 2]"""
    return 10.0 ** np.clip(np.random.default_rng(seed).normal(0.0, 0.7, n), -2.0, 2.0)


def build(name):
    """(seqs, forms, ess) of one hierarchy"""
    if name == "deformed":
        return amge.build_hierarchy((16, 16, 16), 4, jstart=0, deform=amge.weak_scaling_deformation)[1], (0, 1, 2), ESS_DEFORMED
    if name == "tets":
        V, T, B, A = tets.load_npz(MESH)
        return tets.build_hierarchy(tets.TetMesh(V, T, B, A), 2, 3)[1], (0,), ESS_ALL
    if name == "coefficients":
        nel = 16 ** 3
        seqs = amge.build_hierarchy((16, 16, 16), 4, jstart=0, alpha=lognormal(nel, 1), beta=lognormal(nel, 2))[1]
        return seqs, (1, 2), ESS_ALL
    if name == "uniform8":
        return amge.build_hierarchy((8, 8, 8), 3)[1], (0, 1, 2), ESS_ALL
    raise KeyError(name)


def tridiagonal(n=1000, seed=3):
    """1-D operator with 3 entries per row and random SPD values.  No level operator of the hierarchies above has a
    colour whose rows all hold <= 4 entries, so this is the input of the single-group G = 4 Gauss-Seidel variant."""
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    off = -rng.uniform(0.5, 1.5, n - 1)
    d = np.abs(np.concatenate([off, [0.0]])) + np.abs(np.concatenate([[0.0], off])) + rng.uniform(0.1, 1.0, n)
    A = sp.diags([off, d, off], [-1, 0, 1], format="csr")
    A.sort_indices()
    return A


def level_operators(seqs, form, ess):
    """[(label, matrix)]: A_l of every level (Galerkin, FixZeroRows) and, for forms > 0, the Hiptmair auxiliary
    operator fix_zero_rows(D_l^T A_l D_l) of every level"""
    A, _ = drivers.system_matrix(seqs[0], form, ess)
    out = []
    for l in range(len(seqs)):
        if l > 0:
            A, _ = orc.fix_zero_rows(orc.rap(A, seqs[l - 1].get_P(form, ess)))
        out.append(("L%d-A" % l, A))
        if form > 0:
            Aaux, _ = orc.fix_zero_rows(orc.rap(A, seqs[l].get_D(form - 1, ess)))
            out.append(("L%d-aux" % l, Aaux))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# predictor
# ---------------------------------------------------------------------------------------------------------------------
def pick_group(wmax, forced=0):
    """pe_sell.cu sell_pick_group: (G, single)"""
    if forced in GROUPS:
        G = forced
    elif wmax <= 4:
        G = 4
    elif wmax <= 8:
        G = 8
    elif wmax <= 12:
        G = 12
    elif wmax <= 24:
        G = 8
    else:
        G = 4
    return G, wmax <= G


def slice_widths(lens):
    """widths of the slices of 32 consecutive rows of the given lengths (last slice padded)"""
    lens = np.asarray(lens, dtype=np.int64)
    pad = np.zeros(-len(lens) % 32, dtype=np.int64)
    return np.concatenate([lens, pad]).reshape(-1, 32).max(axis=1)


def colour_layout(A):
    """(order, set_starts, [(slices, widest slice)] per colour) of the colour-ordered SELL copy"""
    color, ncol = orc.greedy_colors(A)
    order = np.argsort(color, kind="stable").astype(np.int32)
    starts = np.concatenate([[0], np.cumsum(np.bincount(color, minlength=ncol))]).astype(np.int64)
    lens = np.diff(A.indptr)[order]
    per = []
    for c in range(ncol):
        w = slice_widths(lens[starts[c]:starts[c + 1]])
        per.append((len(w), int(w.max()) if len(w) else 0))
    return order, starts, per


def skips_turn(A, order, starts):
    """build_gs_schedule: the backward pass of l1-GS skips the last colour when l1 == a_ii > 0 on all of its rows"""
    if len(starts) < 3:
        return False
    l1 = orc.l1_norms(A, 2)
    d = A.diagonal()
    rows = order[starts[-2]:starts[-1]]
    return bool(np.all((d[rows] > 0.0) & (l1[rows] == d[rows])))


def gs_counts(A, forced=0, sweeps=2, zero_guess=False, skip_turn=None):
    """{(G, single): padded slice rows} of one multicolour l1-GS application on the SELL path"""
    order, starts, per = colour_layout(A)
    if skip_turn is None:
        skip_turn = skips_turn(A, order, starts)
    ncol = len(per)
    out = dict.fromkeys(CHOICES, 0)
    for sweep in range(sweeps):
        first = -1
        if zero_guess and sweep == 0:
            first = next(c for c in range(ncol) if per[c][0] > 0 or c == ncol - 1)
        for p in range(2):
            for cc in range(1 if (p == 1 and skip_turn) else 0, ncol):
                c = cc if p == 0 else ncol - 1 - cc
                nsl, w = per[c]
                if nsl == 0 or (p == 0 and c == first):
                    continue
                out[pick_group(w, forced)] += 32 * nsl
    return out


def spmv_choice(A, forced=0):
    """(G, single, padded slice rows) of a SELL SpMV with A, or None when A takes another kernel"""
    w = slice_widths(np.diff(A.indptr))
    if A.nnz == 0 or 32 * w.sum() > 1.25 * A.nnz:
        return None
    G, single = pick_group(int(w.max()), forced)
    return G, single, 32 * len(w)


def report(name, forced_groups=(0, 4, 8, 12)):
    """{forced group: {(G, single): padded slice rows}} of one sweep (2 sweeps, iterative mode) on every level operator
    of every form of one hierarchy"""
    seqs, forms, ess = build(name)
    out = {g: dict.fromkeys(CHOICES, 0) for g in forced_groups}
    for form in forms:
        for _, A in level_operators(seqs, form, ess):
            for g in forced_groups:
                for k, v in gs_counts(A, forced=g).items():
                    out[g][k] += v
    return out
