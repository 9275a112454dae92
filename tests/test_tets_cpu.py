"""Tetrahedral meshes (BASELINE configs[0]: examples/MultigridTest0Form.cpp on meshes/cube456.mesh), CPU side: the product's
host code (parelag_b200/src/amge_tet.hpp: mesh reader, red refinement, topology, Whitney mass matrices, targets) against the
oracle (oracle/tets.py); integer tables bit-exact, values to 1e-13; and the oracle itself against the CheckInvariants
identities (DeRhamSequence.cpp:694-970) and the dof counts SURVEY 8(d) quotes for configs[0].
tests/golden/cube456.npz holds the arrays of the reference's input mesh meshes/cube456.mesh (written by
tests/golden/make_cube456.py from that file), so the tests need nothing outside the repository."""
import os

import numpy as np
import pytest

from parelag_b200 import api
from oracle import amge, drivers, tets

MESH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cube456.npz")


def same(A, B):
    A.sort_indices(); B = B.tocsr(); B.sort_indices()
    return (A.shape == B.shape and np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices)
            and np.array_equal(A.data, B.data))


def test_cube456_counts_match_the_reference_configuration():
    """SURVEY 8(d) cfg 1: 141 vertices, 456 tets; after 2 refinements 5 739 H1 dofs (the coarsest level of the driver's
    3-level hierarchy), after 3: 42 309, and the mesh fills the unit cube with 6 boundary attributes."""
    m = tets.TetMesh(*tets.load_npz(MESH))
    assert (m.nv, m.nel) == (141, 456) and abs(m.vol.sum() - 1.0) < 1e-12
    assert abs(m.facet_area()[m.bdr_face].sum() - 6.0) < 1e-12 and sorted(set(m.Battr.tolist())) == [1, 2, 3, 4, 5, 6]
    m2 = m.refine().refine()
    assert (m2.nv, m2.nel) == (5739, 29184)
    m3 = m2.refine()
    assert (m3.nv, m3.nel) == (42309, 233472)
    assert (m3.ne + 0, m3.nf + 0) == (m3.ne, m3.nf) and m3.nv - m3.ne + m3.nf - m3.nel == 1      # Euler characteristic of a ball


def test_oracle_tet_hierarchy_invariants_and_nested_spaces():
    """derefinement of a refined tet mesh reproduces the coarser meshes' entity counts; Whitney spaces are nested, so
    no NullSpace dof appears and the CheckInvariants identities hold"""
    m0 = tets.TetMesh(*tets.cube_tets(1))
    mesh, seqs = tets.build_hierarchy(m0, 2, 3)
    m1 = m0.refine()
    assert [s.dof[0].ndofs for s in seqs] == [mesh.nv, m1.nv, m0.nv]
    assert [s.dof[1].ndofs for s in seqs] == [mesh.ne, m1.ne, m0.ne]
    assert [s.dof[2].ndofs for s in seqs] == [mesh.nf, m1.nf, m0.nf]
    for s in seqs[:-1]:
        amge.check_invariants(s)
        assert all(v in (0, (0, 0)) for v in s.stats.values())


@pytest.mark.parametrize("case", ["kuhn", "cube456"])
def test_product_tet_tables_match_oracle(case):
    if case == "kuhn":
        V, T, B, A = tets.cube_tets(2)
        nref, nlev = 2, 3
    else:
        V, T, B, A = tets.load_npz(MESH)
        nref, nlev = 1, 2
    S = api.Sequence.tet(V, T, B, A, nref, nlev, svd_tol=-1.0)
    mesh = tets.TetMesh(V, T, B, A)
    for _ in range(nref):
        mesh = mesh.refine()
    topo = mesh.topology()
    seq = tets.fine_sequence_tet(mesh, topo)
    n = mesh.nel
    t = topo
    for l in range(nlev):
        for c in range(3):
            assert same(S.get_csr(l, "B", c), t.B[c]), (l, c)
        assert same(S.get_csr(l, "FB"), t.facet_bdr)
        if l + 1 < nlev:
            ct = t.coarsen(np.arange(n) // 8)
            for c in range(4):
                assert same(S.get_csr(l, "AE", c), t.AE_entity[c]), (l, c)
            t, n = ct, n // 8
    for j in range(3):
        assert same(S.get_csr(0, "D", j), seq.D[j]) if j < 2 else abs(S.get_csr(0, "D", j) - seq.D[j]).max() <= 1e-13 * abs(seq.D[j]).max()
    for j in range(4):
        for c in range(4 - j):
            Me, Mo = S.get_csr(0, "Me", j, c), seq.M[(j, c)]
            assert Me.shape == Mo.shape and abs(Me - Mo).max() <= 1e-13 * abs(Mo).max(), (j, c)
            assert same(S.get_csr(0, "ED", j, c), seq.dof[j].entity_dof[c])
        Tg, To = S.get_targets(0, j), seq.targets[j]
        assert np.abs(Tg - To).max() <= 1e-14 * max(np.abs(To).max(), 1.0)
        assert np.array_equal(S.get_bdr_mask(0, j), drivers.bdr_mask(seq.dof[j]))
    S.free()


def test_product_reads_the_mesh_file(tmp_path):
    """the product's NETGEN-neutral reader (what mfem::Mesh(imesh, 1, 1) does at examples/MultigridTest0Form.cpp:139-148):
    the arrays are written in that format (and re-read by the oracle's reader), the product reads the file"""
    V, T, B, A = tets.load_npz(MESH)
    path = str(tmp_path / "cube456.mesh")
    tets.write_netgen_neutral(path, V, T, B, A)
    V2, T2, B2, A2 = tets.read_netgen_neutral(path)
    assert np.array_equal(V2, V) and np.array_equal(T2, T) and np.array_equal(B2, B) and np.array_equal(A2, A)
    S = api.Sequence.tet_from_file(path, 0, 1, svd_tol=-1.0)
    m = tets.TetMesh(V, T, B, A)
    topo = m.topology()
    assert same(S.get_csr(0, "B", 0), topo.B[0]) and same(S.get_csr(0, "FB"), topo.facet_bdr)
    assert np.array_equal(S.get_targets(0, 0)[:, 3], V[:, 0])        # vertex coordinates survive the round trip bit for bit
    S.free()


def test_product_reads_the_mfem_mesh_format(tmp_path):
    """MFEM's own "MFEM mesh v1.0" format (comment block, 0-based vertices, geometry types): recognised from the first line
    like mfem::Mesh(imesh, 1, 1); same tables as from the arrays; unsupported content is refused"""
    from parelag_b200 import capi
    V, T, B, A = tets.load_npz(MESH)
    path = str(tmp_path / "cube456_mfem.mesh")
    tets.write_mfem_mesh(path, V, T, B, A)
    V2, T2, B2, A2 = tets.read_mfem_mesh(path)
    assert np.array_equal(V2, V) and np.array_equal(T2, T) and np.array_equal(B2, B) and np.array_equal(A2, A)
    S = api.Sequence.tet_from_file(path, 0, 1, svd_tol=-1.0)
    R = api.Sequence.tet(V, T, B, A, 0, 1, svd_tol=-1.0)
    for c in range(3):
        assert same(S.get_csr(0, "B", c), R.get_csr(0, "B", c))
    assert same(S.get_csr(0, "FB"), R.get_csr(0, "FB"))
    assert np.array_equal(S.get_targets(0, 0), R.get_targets(0, 0))
    for j in range(4):
        assert abs(S.get_csr(0, "Me", j, 0) - R.get_csr(0, "Me", j, 0)).max() == 0
    S.free(); R.free()
    bad = str(tmp_path / "hex.mesh")
    open(bad, "w").write("MFEM mesh v1.0\n\ndimension\n3\n\nelements\n1\n1 5 0 1 2 3 4 5 6 7\n\nboundary\n0\n\nvertices\n8\n3\n" + "0 0 0\n" * 8)
    with pytest.raises(capi.PEError, match="only tetrahedra"):
        api.Sequence.tet_from_file(bad, 0, 1, svd_tol=-1.0)
