"""Colour-numbered V-cycle levels (Hierarchy::SetupColour): a level whose smoother is multicolour SELL Gauss-Seidel keeps
its vectors in the smoother's colour numbering for the whole cycle, so its products run on renumbered copies
(pe_mat_renumbered) and the smoother runs without renumbering passes (pe_smoother_apply_colour).  Checked here, on the
uniform and the irregular hierarchies with PE_TUNE_SELL_MIN_ROWS = 0 so that every level takes SELL:
  a. every renumbered product -- residual, P^T, P with beta = 1, D^T, D with beta = 1 -- equals the natural product
     followed by the permutation, bit for bit, and leaves the padding entries 0;
  b. the colour-numbered smoother forms (zero guess, initial guess, entry pass + sweep + exit pass) equal the natural
     pe_smoother_apply bit for bit.
The whole cycle in direct, graph and program mode against the oracle is tests/test_vcycle_modes_gpu.py and
tests/test_vcycle_irregular_gpu.py, which run these levels colour-numbered."""
import numpy as np
import pytest

from parelag_b200 import api, capi
from tests import irregular_hierarchies as IH
from tests.test_vcycle_modes_gpu import tuning

pytestmark = pytest.mark.gpu

CASES = [("uniform8", 2), ("deformed", 1), ("coefficients", 2), ("tets", 0)]


@pytest.fixture(scope="module")
def sess():
    return api.session()


@pytest.fixture(scope="module")
def hiers():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = IH.build(name)
        return cache[name]
    return get


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


class Numbered:
    """a multicolour l1-GS smoother on A and its colour numbering: host pos (row -> position), npad, device pos"""

    def __init__(self, sess, A, sweeps=1):
        self.M = capi.Mat.from_scipy(sess, A)
        self.S = capi.Smoother(sess, self.M, type=2, sweeps=sweeps, ordering=capi.GS_MULTICOLOR)
        self.npad, self.pos_d = self.S.colour_numbering()
        assert self.npad > 0, "the SELL path with a colour numbering was expected"
        order, starts = self.S.order()
        self.pos = np.empty(len(order), dtype=np.int64)
        slice0 = 0
        for c in range(len(starts) - 1):
            rows = order[starts[c]:starts[c + 1]]
            self.pos[rows] = 32 * slice0 + np.arange(len(rows))
            slice0 += (len(rows) + 31) // 32
        assert self.npad == 32 * slice0

    def to_colour(self, x):
        out = np.zeros(self.npad)
        out[self.pos] = x
        return out

    def padding(self, xc):
        mask = np.ones(self.npad, dtype=bool)
        mask[self.pos] = False
        return xc[mask]

    def free(self):
        self.S.free(); self.M.free()


def natural_product(sess, M, x, y0=None, transpose=False, residual_b=None):
    nr = M.info()[1] if transpose else M.info()[0]
    dx, dy = capi.Vec(sess, data=x), capi.Vec(sess, data=np.zeros(nr) if y0 is None else y0)
    if residual_b is not None:
        db = capi.Vec(sess, data=residual_b)
        M.residual(dx, db, dy)
        db.free()
    elif transpose:
        M.spmv_t(dx, dy, 1.0, 0.0 if y0 is None else 1.0)
    else:
        M.spmv(dx, dy, 1.0, 0.0 if y0 is None else 1.0)
    out = dy.download()
    dx.free(); dy.free()
    return out


def renumbered_product(sess, R, x, nrows_out, y0=None, residual_b=None):
    dx, dy = capi.Vec(sess, data=x), capi.Vec(sess, data=np.zeros(nrows_out) if y0 is None else y0)
    if residual_b is not None:
        db = capi.Vec(sess, data=residual_b)
        R.residual(dx, db, dy)
        db.free()
    else:
        R.spmv(dx, dy, 1.0, 0.0 if y0 is None else 1.0)
    out = dy.download()
    dx.free(); dy.free()
    return out


@pytest.mark.parametrize("name,form", CASES, ids=["%s-form%d" % c for c in CASES])
def test_renumbered_products_are_the_permuted_natural_products(sess, hiers, name, form):
    seqs, _, ess = hiers(name)
    ops = dict(IH.level_operators(seqs, form, ess))
    rng = np.random.default_rng(7)
    with tuning(SELL_MIN_ROWS=0, FUSED_GS_MAX_MB=0):
        for l in range(len(seqs) - 1):
            A, Ac = ops["L%d-A" % l], ops["L%d-A" % (l + 1)]
            f, c = Numbered(sess, A), Numbered(sess, Ac)
            MA = capi.Mat.from_scipy(sess, A)
            x, b = rng.standard_normal(A.shape[0]), rng.standard_normal(A.shape[0])
            # residual b - A x, colour <- colour
            R = MA.renumbered(False, f.pos_d, f.npad, f.pos_d, f.npad)
            got = renumbered_product(sess, R, f.to_colour(x), f.npad, residual_b=f.to_colour(b))
            ref = natural_product(sess, MA, x, residual_b=b)
            assert np.array_equal(bits(got[f.pos]), bits(ref)), (l, "residual")
            assert not np.any(f.padding(got)), (l, "residual padding")
            R.free()
            # P^T (coarse colour <- fine colour), P with beta = 1 (fine colour <- coarse colour); P as in the hierarchy
            P = seqs[l].get_P(form, ess)
            MP = capi.Mat.from_scipy(sess, P)
            for (rows, cols) in ((c, f), (None, f), (c, None)):
                Rt = MP.renumbered(True, rows and rows.pos_d, rows.npad if rows else 0, cols and cols.pos_d, cols.npad if cols else 0)
                got = renumbered_product(sess, Rt, cols.to_colour(x) if cols else x, rows.npad if rows else P.shape[1])
                ref = natural_product(sess, MP, x, transpose=True)
                assert np.array_equal(bits(got[rows.pos] if rows else got), bits(ref)), (l, "P^T")
                if rows:
                    assert not np.any(rows.padding(got)), (l, "P^T padding")
                Rt.free()
            e, y0 = rng.standard_normal(P.shape[1]), rng.standard_normal(P.shape[0])
            Rp = MP.renumbered(False, f.pos_d, f.npad, c.pos_d, c.npad)
            got = renumbered_product(sess, Rp, c.to_colour(e), f.npad, y0=f.to_colour(y0))
            ref = natural_product(sess, MP, e, y0=y0)
            assert np.array_equal(bits(got[f.pos]), bits(ref)), (l, "P beta=1")
            assert not np.any(f.padding(got)), (l, "P padding")
            Rp.free(); MP.free()
            if form > 0:
                # Hiptmair: D^T (auxiliary colour <- primary colour), D with beta = 1 (primary colour <- auxiliary colour)
                D = seqs[l].get_D(form - 1, ess)
                a = Numbered(sess, ops["L%d-aux" % l])
                MD = capi.Mat.from_scipy(sess, D)
                Rdt = MD.renumbered(True, a.pos_d, a.npad, f.pos_d, f.npad)
                got = renumbered_product(sess, Rdt, f.to_colour(x), a.npad)
                ref = natural_product(sess, MD, x, transpose=True)
                assert np.array_equal(bits(got[a.pos]), bits(ref)), (l, "D^T")
                assert not np.any(a.padding(got)), (l, "D^T padding")
                z = rng.standard_normal(D.shape[1])
                Rd = MD.renumbered(False, f.pos_d, f.npad, a.pos_d, a.npad)
                got = renumbered_product(sess, Rd, a.to_colour(z), f.npad, y0=f.to_colour(y0))
                ref = natural_product(sess, MD, z, y0=y0)
                assert np.array_equal(bits(got[f.pos]), bits(ref)), (l, "D beta=1")
                assert not np.any(f.padding(got)), (l, "D padding")
                Rdt.free(); Rd.free(); MD.free(); a.free()
            MA.free(); f.free(); c.free()


@pytest.mark.parametrize("name,form", CASES, ids=["%s-form%d" % c for c in CASES])
@pytest.mark.parametrize("sweeps", [1, 2])
def test_colour_smoother_forms_match_the_natural_smoother(sess, hiers, name, form, sweeps):
    seqs, _, ess = hiers(name)
    rng = np.random.default_rng(11)
    with tuning(SELL_MIN_ROWS=0, FUSED_GS_MAX_MB=0):
        for lab, A in IH.level_operators(seqs, form, ess):
            s = Numbered(sess, A, sweeps)
            S = s.S
            n = A.shape[0]
            b, x0 = rng.standard_normal(n), rng.standard_normal(n)

            def natural(iterative):
                db, dx = capi.Vec(sess, data=b), capi.Vec(sess, data=x0 if iterative else np.full(n, 7.0))
                S.apply(db, dx, iterative)
                out = dx.download()
                db.free(); dx.free()
                return out

            fc = capi.Vec(sess, data=s.to_colour(b))
            for mode, start in ((0, s.to_colour(x0)), (1, np.full(s.npad, 7.0))):
                uc = capi.Vec(sess, data=start)
                S.apply_colour(fc, uc, mode)
                got = uc.download()
                assert np.array_equal(bits(got[s.pos]), bits(natural(mode == 0))), (lab, mode)
                if mode == 1:
                    assert not np.any(s.padding(got)), (lab, "padding")
                uc.free()
            # entry pass (renumbering + first colour), sweep, exit pass == the natural smoother from a zero guess
            db, f2, u2, x = capi.Vec(sess, data=b), capi.Vec(sess, s.npad), capi.Vec(sess, s.npad), capi.Vec(sess, n)
            S.colour_in(db, f2, u2)
            assert np.array_equal(bits(f2.download()), bits(s.to_colour(b))), lab
            S.apply_colour(f2, u2, 2)
            S.colour_out(u2, x)
            assert np.array_equal(bits(x.download()), bits(natural(False))), (lab, "in/out")
            for v in (db, f2, u2, x, fc):
                v.free()
            s.free()
