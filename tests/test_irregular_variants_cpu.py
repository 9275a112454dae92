"""Which entry-group variants of the SELL Gauss-Seidel kernel (k_sell_gs<G, SINGLE>) the irregular hierarchies of
tests/test_vcycle_irregular_gpu.py reach, from the host rules alone (tests/irregular_hierarchies.py); no GPU."""
import numpy as np
import pytest

from tests import irregular_hierarchies as IH


def reached(report):
    return {g: {k for k, v in counts.items() if v > 0} for g, counts in report.items()}


@pytest.fixture(scope="module")
def reports():
    return {name: IH.report(name) for name in ("uniform8", "deformed", "coefficients")}


def test_pick_group_rule():
    auto = {w: IH.pick_group(w) for w in (1, 4, 5, 8, 9, 12, 13, 24, 25, 137)}
    assert auto == {1: (4, True), 4: (4, True), 5: (8, True), 8: (8, True), 9: (12, True), 12: (12, True),
                    13: (8, False), 24: (8, False), 25: (4, False), 137: (4, False)}
    # forced sizes: single-group exactly when the widest slice fits one group
    for G in IH.GROUPS:
        assert IH.pick_group(G, G) == (G, True) and IH.pick_group(G + 1, G) == (G, False)
    # G = 12 pipelined is only ever a forced choice
    assert all(IH.pick_group(w) != (12, False) for w in range(1, 400))


def test_colour_layout_and_counts_of_a_small_operator():
    """hand-checked: the 1-D operator has two colours (even, odd rows), 500 rows each -> 16 slices of width <= 3"""
    A = IH.tridiagonal(1000)
    order, starts, per = IH.colour_layout(A)
    assert list(starts) == [0, 500, 1000] and np.array_equal(order[:500], np.arange(0, 1000, 2))
    assert per == [(16, 3), (16, 3)]
    # l1 == diagonal on the last colour: the backward pass starts with colour 0; 2 sweeps x 3 colour launches
    expected = dict.fromkeys(IH.CHOICES, 0)
    expected[(4, True)] = 2 * 3 * 16 * 32
    assert IH.gs_counts(A) == expected
    # zero initial guess: the first colour of the first forward pass is folded into the renumbering
    assert IH.gs_counts(A, zero_guess=True)[(4, True)] == (2 * 3 - 1) * 16 * 32
    assert IH.gs_counts(A, forced=12)[(12, True)] == 2 * 3 * 16 * 32
    assert IH.spmv_choice(A) == (4, True, 32 * 32)


def test_irregular_hierarchies_reach_every_gs_choice(reports):
    """Union over the deformed and the variable-coefficient hierarchies, automatic (0) and forced (4, 8, 12) group
    sizes, plus the 1-D operator for the single-group G = 4 variant: all six (G, single) choices of k_sell_gs run."""
    seen = set()
    for name in ("deformed", "coefficients"):
        for g, keys in reached(reports[name]).items():
            seen.update(keys)
    assert seen == set(IH.CHOICES) - {(4, True)}, sorted(seen)
    assert IH.gs_counts(IH.tridiagonal())[(4, True)] > 0
    # the deformed hierarchy alone: rows of 90-137 entries take pipelined G = 4, ragged coarse rows G = 8 pipelined
    assert reached(reports["deformed"])[0] == {(4, False), (8, False), (12, True)}
    # G = 12 pipelined only when forced
    assert all(reports[n][0][(12, False)] == 0 and reports[n][12][(12, False)] > 0 for n in reports)


def test_uniform_fixture_report(reports):
    """The uniform 8^3 hierarchy of the other V-cycle tests reaches four of the six choices automatically; it never
    reaches the single-group G = 4 variant (it has no rows of <= 4 entries)."""
    r = reached(reports["uniform8"])
    assert r[0] == {(4, False), (8, True), (8, False), (12, True)}
    assert r[4] == {(4, False)} and r[8] == {(8, True), (8, False)} and r[12] == {(12, True), (12, False)}
