"""ctypes binding of include/parelag_b200_api.h: the ParameterList-driven solver API
(SolverLibrary -> SolverFactory -> BuildSolver -> Mult) and the DeRhamSequence
operator interface, as a ParElag driver uses them."""
import ctypes as C

import numpy as np

from . import capi
from .capi import _chk, _ptr, _i32, _f64, lib


def session(rank=0, nranks=1, device=0, nccl_id=None):
    _chk(lib().pe_api_session_create(rank, nranks, device, nccl_id))
    lib().pe_api_session_ctx.restype = C.c_void_p
    ctx = capi.Ctx.__new__(capi.Ctx)
    ctx.h = C.c_void_p(lib().pe_api_session_ctx())
    ctx.close = lambda: None          # owned by the session
    return ctx


def session_destroy():
    _chk(lib().pe_api_session_destroy())


_host_comm = None


def set_host_comm(comm):
    """Install the setup-time host communicator (parelag_b200.par.HostComm); kept alive here."""
    global _host_comm
    _host_comm = comm
    _chk(lib().pe_api_session_set_host_comm(comm.ptr()))


def set_topology_options(partitioner="derefine", check_topology=False, element_partitioning=None):
    """process-wide options of the topology coarsening inside the sequence builders: partitioner "derefine" (default),
    "geometric" (GeometricBoxPartitioner), "user" (element_partitioning as given; two levels) or "logical"
    (LogicalPartitioner; element_partitioning = material id of every fine element); check_topology = second
    argument of CoarsenLocalPartitioning.  Clears the topology log."""
    kind = {"derefine": 0, "geometric": 1, "user": 2, "logical": 3}[partitioner]
    part = None if element_partitioning is None else _i32(element_partitioning)
    _chk(lib().pe_api_set_topology_options(kind, int(bool(check_topology)), _ptr(part), 0 if part is None else len(part)))


def spe10_read(path, N=(60, 220, 85), h=(20.0, 10.0, 2.0)):
    """InversePermeabilityFunction::SetNumberCells / SetMeshSizes / ReadPermeabilityFile"""
    _chk(lib().pe_api_spe10_read(str(path).encode(), N[0], N[1], N[2], C.c_double(h[0]), C.c_double(h[1]), C.c_double(h[2])))


def spe10_data():
    n = C.c_int64()
    _chk(lib().pe_api_spe10_data(None, C.byref(n)))
    out = np.empty(n.value)
    _chk(lib().pe_api_spe10_data(_ptr(out), None))
    return out


def spe10_inverse_permeability(x):
    x = _f64(np.ascontiguousarray(x).reshape(-1, 3))
    out = np.empty_like(x)
    _chk(lib().pe_api_spe10_inverse_permeability(_ptr(x), len(x), _ptr(out)))
    return out


def _lines(fn, *args):
    need = C.c_int64()
    _chk(fn(*args, None, C.c_int64(0), C.byref(need)))
    buf = C.create_string_buffer(need.value)
    _chk(fn(*args, buf, C.c_int64(need.value), None))
    return [l for l in buf.value.decode().split("\n") if l]


def parameterlist_dump(xml):
    """the parsed XML parameter list, one "path/name<TAB>type<TAB>value" line per parameter, sorted"""
    return _lines(lib().pe_api_parameterlist_dump, xml.encode())


def library_factories(xml):
    """[(solver name, factory type, "ok" | "error: ...")] for every entry of the document's Preconditioner Library"""
    return [tuple(l.split("\t", 2)) for l in _lines(lib().pe_api_library_factories, xml.encode())]


def topology_log():
    """the lines the reference prints during the topology coarsening (since the options were last set)"""
    need = C.c_int64()
    _chk(lib().pe_api_topology_log(None, C.c_int64(0), C.byref(need)))
    buf = C.create_string_buffer(need.value)
    _chk(lib().pe_api_topology_log(buf, C.c_int64(need.value), None))
    return [l for l in buf.value.decode().split("\n") if l]


def _csr_args(M):
    M = M.tocsr()
    return (M.shape[0], M.shape[1], np.ascontiguousarray(M.indptr, dtype=np.int32),
            np.ascontiguousarray(M.indices, dtype=np.int32), np.ascontiguousarray(M.data, dtype=np.float64))


class Sequence:
    """A chain of DeRhamSequence levels with supplied operators."""

    def __init__(self, nforms, nlevels):
        self.h = C.c_void_p()
        _chk(lib().pe_api_sequence_create(nforms, nlevels, C.byref(self.h)))

    def set_P(self, level, form, P):
        nr, nc, I, J, A = _csr_args(P)
        _chk(lib().pe_api_sequence_set_P(self.h, level, form, nr, nc, _ptr(I), _ptr(J), _ptr(A)))

    def set_D(self, level, form, D):
        nr, nc, I, J, A = _csr_args(D)
        _chk(lib().pe_api_sequence_set_D(self.h, level, form, nr, nc, _ptr(I), _ptr(J), _ptr(A)))

    def set_bdr_mask(self, level, form, mask):
        mask = np.ascontiguousarray(mask, dtype=np.uint32)
        _chk(lib().pe_api_sequence_set_bdr_mask(self.h, level, form, len(mask), _ptr(mask)))

    @staticmethod
    def hex(dims, nlevels, L=(1.0, 1.0, 1.0), alpha=None, beta=None, jstart=0, svd_tol=1e-9, coords=None):
        """Full coarsening path on a structured hex mesh (svd_tol < 0: topology only).  coords: optional (nv, 3)
        moved vertices (trilinear hexahedra, index-grid numbering)."""
        S = Sequence.__new__(Sequence)
        S.h = C.c_void_p()
        a = None if alpha is None else _f64(alpha)
        b = None if beta is None else _f64(beta)
        if coords is not None:
            X = _f64(np.ascontiguousarray(coords).ravel())
            _chk(lib().pe_api_hexsequence_create_deformed(dims[0], dims[1], dims[2], _ptr(X), _ptr(a), _ptr(b), jstart, nlevels,
                                                          C.c_double(svd_tol), C.byref(S.h)))
            return S
        _chk(lib().pe_api_hexsequence_create(dims[0], dims[1], dims[2], C.c_double(L[0]), C.c_double(L[1]),
                                             C.c_double(L[2]), _ptr(a), _ptr(b), jstart, nlevels,
                                             C.c_double(svd_tol), C.byref(S.h)))
        return S

    @staticmethod
    def hex_tensor(dims, nlevels, beta_xyz, L=(1.0, 1.0, 1.0), alpha=None, jstart=0, svd_tol=1e-9):
        """hex() with a diagonal tensor coefficient in the H(div) mass matrices: beta_xyz (nel, 3)"""
        S = Sequence.__new__(Sequence)
        S.h = C.c_void_p()
        a = None if alpha is None else _f64(alpha)
        b = _f64(np.ascontiguousarray(beta_xyz).reshape(-1))
        assert len(b) == 3 * dims[0] * dims[1] * dims[2]
        _chk(lib().pe_api_hexsequence_create_tensor(dims[0], dims[1], dims[2], C.c_double(L[0]), C.c_double(L[1]), C.c_double(L[2]),
                                                    _ptr(a), _ptr(b), jstart, nlevels, C.c_double(svd_tol), C.byref(S.h)))
        return S

    @staticmethod
    def spe10(dims, h, nlevels, jstart=2, svd_tol=1e-9):
        """the mesh of examples/MultigridTestSPE10.cpp (dims cells of size h) with the loaded SPE10 inverse permeability
        (spe10_read) as the tensor coefficient of the H(div) mass matrix"""
        S = Sequence.__new__(Sequence)
        S.h = C.c_void_p()
        _chk(lib().pe_api_hexsequence_create_spe10(dims[0], dims[1], dims[2], C.c_double(h[0]), C.c_double(h[1]), C.c_double(h[2]),
                                                   jstart, nlevels, C.c_double(svd_tol), C.byref(S.h)))
        return S

    @staticmethod
    def tet(V, T, Btri, Battr, nref, nlevels, jstart=0, svd_tol=1e-9):
        """Full coarsening path on a tetrahedral mesh refined nref times (V: (nv,3); T: (nel,4) 0-based; Btri: (nb,3);
        Battr: (nb,) 1-based boundary attributes); svd_tol < 0: topology and fine sequence only."""
        S = Sequence.__new__(Sequence)
        S.h = C.c_void_p()
        X, Tt, Bt, Ba = _f64(np.ascontiguousarray(V).ravel()), _i32(np.ascontiguousarray(T).ravel()), _i32(np.ascontiguousarray(Btri).ravel()), _i32(Battr)
        _chk(lib().pe_api_tetsequence_create(len(X) // 3, _ptr(X), len(Tt) // 4, _ptr(Tt), len(Ba), _ptr(Bt), _ptr(Ba), nref, nlevels, jstart,
                                             C.c_double(svd_tol), C.byref(S.h)))
        return S

    @staticmethod
    def tet_from_file(path, nref, nlevels, jstart=0, svd_tol=1e-9):
        S = Sequence.__new__(Sequence)
        S.h = C.c_void_p()
        _chk(lib().pe_api_tetsequence_create_from_file(path.encode(), nref, nlevels, jstart, C.c_double(svd_tol), C.byref(S.h)))
        return S

    @staticmethod
    def hex_par(procs, dims, nlevels, L=(1.0, 1.0, 1.0), alpha=None, beta=None, jstart=0, svd_tol=1e-9, coords=None):
        """The same on THIS rank's box (dims hexahedra of extent L) of a procs[0] x procs[1] x procs[2] box
        decomposition; needs set_host_comm().  coords: optional (nv, 3) moved vertices of this rank's box."""
        S = Sequence.__new__(Sequence)
        S.h = C.c_void_p()
        a = None if alpha is None else _f64(alpha)
        b = None if beta is None else _f64(beta)
        P = _i32(procs)
        if coords is not None:
            X = _f64(np.ascontiguousarray(coords).ravel())
            _chk(lib().pe_api_hexsequence_create_par_deformed(_ptr(P), dims[0], dims[1], dims[2], _ptr(X), _ptr(a), _ptr(b),
                                                              jstart, nlevels, C.c_double(svd_tol), C.byref(S.h)))
            return S
        _chk(lib().pe_api_hexsequence_create_par(_ptr(P), dims[0], dims[1], dims[2], C.c_double(L[0]), C.c_double(L[1]),
                                                 C.c_double(L[2]), _ptr(a), _ptr(b), jstart, nlevels,
                                                 C.c_double(svd_tol), C.byref(S.h)))
        return S

    def dofmap(self, level, form):
        """DofHandler::GetDofTrueDof: dict(gid, owner, key, start, ntrue, nglobal) of the local dofs"""
        nd, st, nt, ng = C.c_int32(), C.c_int64(), C.c_int64(), C.c_int64()
        _chk(lib().pe_api_sequence_get_dofmap(self.h, level, form, C.byref(nd), None, None, None, C.byref(st), C.byref(nt), C.byref(ng)))
        gid, owner, key = np.empty(nd.value, dtype=np.int64), np.empty(nd.value, dtype=np.int32), np.empty(nd.value, dtype=np.int64)
        _chk(lib().pe_api_sequence_get_dofmap(self.h, level, form, None, _ptr(gid), _ptr(owner), _ptr(key), None, None, None))
        return dict(gid=gid, owner=owner, key=key, start=st.value, ntrue=nt.value, nglobal=ng.value)

    def assemble_vector(self, level, form, local):
        """SharingMap::Assemble: local dof vector -> true dof vector (copies summed on the owner)"""
        m = self.dofmap(level, form)
        x, out = _f64(local), np.empty(m["ntrue"])
        _chk(lib().pe_api_sequence_dofmap_apply(self.h, level, form, 0, _ptr(x), _ptr(out)))
        return out

    def distribute_vector(self, level, form, true):
        """SharingMap::Distribute: true dof vector -> local dof vector"""
        m = self.dofmap(level, form)
        x, out = _f64(true), np.empty(len(m["gid"]))
        _chk(lib().pe_api_sequence_dofmap_apply(self.h, level, form, 1, _ptr(x), _ptr(out)))
        return out

    def true_operator(self, ctx, level, what, form, ess_attr=None):
        """ComputeTrueP / ComputeTrueD (what = "P" | "D") as a device ParCSR matrix"""
        ess = None if ess_attr is None else _i32(ess_attr)
        m = capi.Mat(ctx)
        _chk(lib().pe_api_sequence_true_operator(self.h, level, what.encode(), form, _ptr(ess), 0 if ess is None else len(ess),
                                                 C.byref(m.h)))
        return m

    def get_csr(self, level, what, a=0, b=0):
        import scipy.sparse as sp
        nr, nc, nnz = C.c_int32(), C.c_int32(), C.c_int64()
        _chk(lib().pe_api_sequence_get_csr(self.h, level, what.encode(), a, b, C.byref(nr), C.byref(nc),
                                           C.byref(nnz), None, None, None))
        I = np.empty(nr.value + 1, dtype=np.int32)
        J = np.empty(nnz.value, dtype=np.int32)
        A = np.empty(nnz.value)
        _chk(lib().pe_api_sequence_get_csr(self.h, level, what.encode(), a, b, None, None, None,
                                           _ptr(I), _ptr(J), _ptr(A)))
        M = sp.csr_matrix((nr.value, nc.value))
        M.data, M.indices, M.indptr = A, J, I
        return M

    def get_targets(self, level, form):
        nd, nt = C.c_int32(), C.c_int32()
        _chk(lib().pe_api_sequence_get_targets(self.h, level, form, C.byref(nd), C.byref(nt), None))
        out = np.empty(nd.value * nt.value)
        _chk(lib().pe_api_sequence_get_targets(self.h, level, form, None, None, _ptr(out)))
        return out.reshape(nt.value, nd.value).T

    def get_bdr_mask(self, level, form):
        nd = C.c_int32()
        _chk(lib().pe_api_sequence_get_bdr_mask(self.h, level, form, C.byref(nd), None))
        m = np.empty(nd.value, dtype=np.uint32)
        _chk(lib().pe_api_sequence_get_bdr_mask(self.h, level, form, None, _ptr(m)))
        return m

    def assemble_system(self, ctx, level, form, ess_attr):
        ess = None if ess_attr is None else _i32(ess_attr)
        m = capi.Mat(ctx)
        _chk(lib().pe_api_sequence_assemble_system(self.h, level, form, _ptr(ess), 0 if ess is None else len(ess),
                                                   C.byref(m.h)))
        return m

    def assemble_darcy(self, ctx, level=0):
        """(M, B, Bt) of the mixed system [[M Bt][B 0]] as device matrices"""
        M, B, Bt = capi.Mat(ctx), capi.Mat(ctx), capi.Mat(ctx)
        _chk(lib().pe_api_sequence_assemble_darcy(self.h, level, C.byref(M.h), C.byref(B.h), C.byref(Bt.h)))
        return M, B, Bt

    def stat(self, level, name):
        v = C.c_int64()
        _chk(lib().pe_api_sequence_get_stat(self.h, level, name.encode(), C.byref(v)))
        return v.value

    def check_invariants(self, level):
        """DeRhamSequence::CheckInvariants of `level` against the next coarser one; raises PEError naming the violated
        identity, returns the largest residual"""
        w = C.c_double()
        _chk(lib().pe_api_sequence_check_invariants(self.h, level, C.byref(w)))
        return w.value

    def show_topology(self, level):
        """AgglomeratedTopology::ShowMe of one level: entity counts and Euler characteristic, as the reference prints them"""
        need = C.c_int64()
        _chk(lib().pe_api_sequence_show_topology(self.h, level, None, C.c_int64(0), C.byref(need)))
        buf = C.create_string_buffer(need.value)
        _chk(lib().pe_api_sequence_show_topology(self.h, level, buf, C.c_int64(need.value), None))
        return [l for l in buf.value.decode().split("\n") if l]

    def free(self):
        if self.h:
            lib().pe_api_sequence_free(self.h)
            self.h = None


def rank_box(procs, rank):
    """box coordinates of a rank in the procs[0] x procs[1] x procs[2] grid (x fastest, amge_par.hpp)"""
    return (rank % procs[0], (rank // procs[0]) % procs[1], rank // (procs[0] * procs[1]))


def box_vertex_coords(procs, rank_coords, dims, deform=None, domain=(1.0, 1.0, 1.0)):
    """Vertices of one box of a procs[0] x procs[1] x procs[2] decomposition of a domain (index-grid numbering, x
    fastest), computed from the GLOBAL vertex index so that copies of an interface vertex are bitwise equal on every
    rank; deform: optional map of the (nv, 3) array (e.g. weak_scaling_deformation)."""
    ax = []
    for a in range(3):
        ng = procs[a] * dims[a]
        ax.append((np.arange(dims[a] + 1, dtype=np.float64) + rank_coords[a] * dims[a]) * (domain[a] / ng))
    k, j, i = np.meshgrid(ax[2], ax[1], ax[0], indexing="ij")
    X = np.stack([i.ravel(), j.ravel(), k.ravel()], axis=1)
    return X if deform is None else deform(X)


def weak_scaling_deformation(X):
    """examples/3DHdivWeakScaling.cpp:148-158: y += exp(z)/2, then x += sin(y)"""
    X = np.array(X, dtype=np.float64)
    X[:, 1] += 0.5 * np.exp(X[:, 2])
    X[:, 0] += np.sin(X[:, 1])
    return X


def library_xml(entries):
    """entries: {name: (type, {param: value})} -> <ParameterList name="Preconditioner Library">"""
    def ptype(v):
        if isinstance(v, bool):
            return "bool", "true" if v else "false"
        if isinstance(v, int):
            return "int", str(v)
        if isinstance(v, float):
            return "double", repr(v)
        if isinstance(v, (list, tuple)):
            return "vector(int)", " ".join(str(int(x)) for x in v)
        return "string", str(v)
    out = ['<ParameterList name="Preconditioner Library">']
    for name, (typ, params) in entries.items():
        out.append('  <ParameterList name="%s">' % name)
        out.append('    <Parameter name="Type" type="string" value="%s"/>' % typ)
        out.append('    <ParameterList name="Solver Parameters">')
        for k, v in params.items():
            t, s = ptype(v)
            out.append('      <Parameter name="%s" type="%s" value="%s"/>' % (k, t, s))
        out.append('    </ParameterList>')
        out.append('  </ParameterList>')
    out.append('</ParameterList>')
    return "\n".join(out)


class Solver:
    def __init__(self, xml, name, A, seq=None, start_level=0, form=0, ess_attr=None):
        ess = None if ess_attr is None else _i32(ess_attr)
        self.h = C.c_void_p()
        if isinstance(A, capi.Mat):      # device-resident operator: ownership passes to the solver
            self.n = A.info()[0]
            _chk(lib().pe_api_solver_build_device(xml.encode(), name.encode(), A.h, None if seq is None else seq.h,
                                                  start_level, form, _ptr(ess), 0 if ess is None else len(ess),
                                                  C.byref(self.h)))
            A.h = None
            return
        A = A.tocsr()
        self.n = A.shape[0]
        keep = [_i32(A.indptr), _i32(A.indices), _f64(A.data)]
        H = capi.ParCSRHost()
        H.global_num_rows = H.num_rows = A.shape[0]
        H.global_num_cols = H.num_cols_diag = A.shape[1]
        H.diag_i, H.diag_j, H.diag_data = [_ptr(a) for a in keep]
        ess = None if ess_attr is None else _i32(ess_attr)
        self.h = C.c_void_p()
        _chk(lib().pe_api_solver_build(xml.encode(), name.encode(), C.byref(H), None if seq is None else seq.h,
                                       start_level, form, _ptr(ess), 0 if ess is None else len(ess), C.byref(self.h)))

    def set_operator(self, A):
        """SetOperator on the built solver: A (capi.Mat) has the held operator's size and sparsity pattern and new
        values.  Ownership of A passes to the solver, also when the call is refused (capi.PEError)."""
        h, A.h = A.h, None
        _chk(lib().pe_api_solver_set_operator(self.h, h))

    def mult(self, b, x0=None):
        b = _f64(b)
        x = np.zeros(self.n) if x0 is None else _f64(x0).copy()
        _chk(lib().pe_api_solver_mult(self.h, _ptr(b), _ptr(x), self.n, 0 if x0 is None else 1))
        return x

    def mult_transpose(self, b, x0=None):
        b = _f64(b)
        x = np.zeros(self.n) if x0 is None else _f64(x0).copy()
        _chk(lib().pe_api_solver_mult_transpose(self.h, _ptr(b), _ptr(x), self.n, 0 if x0 is None else 1))
        return x

    def mult_device(self, b, x, iterative_mode=False):
        _chk(lib().pe_api_solver_mult_device(self.h, b.h, x.h, 1 if iterative_mode else 0))

    def prec_mult_device(self, b, x):
        _chk(lib().pe_api_solver_prec_mult_device(self.h, b.h, x.h))

    def prec_mult_into(self, b, x):
        """Mult of the preconditioner (one AMGe V-cycle) with caller-owned host buffers: H2D, V-cycle, D2H in the call."""
        _chk(lib().pe_api_solver_prec_mult(self.h, _ptr(b), _ptr(x), self.n))

    def mult_into(self, b, x, iterative_mode=False):
        """Mult with caller-owned host buffers (e.g. pinned): H2D of b, D2H into x inside the call."""
        _chk(lib().pe_api_solver_mult(self.h, _ptr(b), _ptr(x), self.n, 1 if iterative_mode else 0))

    def history(self):
        cnt, it, conv = C.c_int(), C.c_int(), C.c_int()
        _chk(lib().pe_api_solver_get_history(self.h, None, 0, C.byref(cnt), C.byref(it), C.byref(conv)))
        h = np.zeros(cnt.value)
        _chk(lib().pe_api_solver_get_history(self.h, _ptr(h), cnt.value, C.byref(cnt), C.byref(it), C.byref(conv)))
        return h, it.value, bool(conv.value)

    def num_levels(self):
        n = C.c_int()
        _chk(lib().pe_api_solver_num_levels(self.h, C.byref(n)))
        return n.value

    def level_info(self, l):
        a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
        _chk(lib().pe_api_solver_level_info(self.h, l, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def program(self):
        """(nops, algorithmic bytes) of the persistent program the V-cycle runs as, or None."""
        h = C.c_void_p()
        _chk(lib().pe_api_solver_program(self.h, C.byref(h)))
        if not h.value:
            return None
        n, b = C.c_int32(), C.c_double()
        _chk(lib().pe_program_info(h, C.byref(n), C.byref(b)))
        return n.value, b.value

    def replay_mode(self):
        """How the last preconditioner-mode V-cycle ran: "direct", "graph" or "program" (capi.REPLAY_*)."""
        m = C.c_int()
        _chk(lib().pe_api_solver_replay_mode(self.h, C.byref(m)))
        return capi.REPLAY_MODE_NAMES[m.value]

    def program_profile(self, ctx):
        """One extra program launch with per-op device timestamps: (types, usec, bytes) arrays."""
        h = C.c_void_p()
        _chk(lib().pe_api_solver_program(self.h, C.byref(h)))
        if not h.value:
            return None
        n = self.program()[0]
        t, us, by = np.empty(n, dtype=np.int32), np.empty(n), np.empty(n)
        _chk(lib().pe_program_profile(ctx.h, h, _ptr(t), _ptr(us), _ptr(by)))
        return t, us, by

    def level_matrix(self, l):
        import scipy.sparse as sp
        n, nnz, _ = self.level_info(l)
        I, J, A = np.empty(n + 1, dtype=np.int32), np.empty(nnz, dtype=np.int32), np.empty(nnz)
        _chk(lib().pe_api_solver_level_matrix(self.h, l, _ptr(I), _ptr(J), _ptr(A)))
        M = sp.csr_matrix((n, n))
        M.data, M.indices, M.indptr = A, J, I
        return M

    def free(self):
        if self.h:
            lib().pe_api_solver_free(self.h)
            self.h = None


class BlockSolver(Solver):
    """BuildSolver on an MfemBlockOperator; blocks: nested list of capi.Mat or None (ownership passes)."""

    def __init__(self, xml, name, blocks, seq, start_level, forms, ess_attr=None):
        nb = len(blocks)
        arr = (C.c_void_p * (nb * nb))()
        self.n = 0
        for i in range(nb):
            h = None
            for j in range(nb):
                b = blocks[i][j]
                arr[i * nb + j] = None if b is None else b.h
                if b is not None and h is None:
                    h = b.info()[0]
            if h is None:
                h = next(blocks[j][i].info()[1] for j in range(nb) if blocks[j][i] is not None)
            self.n += h
        f = _i32(forms)
        ess = None if ess_attr is None else _i32(np.asarray(ess_attr).reshape(nb, -1))
        self.h = C.c_void_p()
        _chk(lib().pe_api_solver_build_block(xml.encode(), name.encode(), nb, arr, None if seq is None else seq.h, start_level,
                                             _ptr(f), _ptr(ess), 0 if ess is None else ess.shape[1], C.byref(self.h)))
        for row in blocks:
            for b in row:
                if b is not None:
                    b.h = None

    def set_blocks(self, blocks):
        """SetOperator on the built block solver: blocks (nested list of capi.Mat or None) have the held operator's zero
        blocks, block sizes and sparsity patterns, and new values.  Ownership passes to the solver, also when the call is
        refused (capi.PEError)."""
        nb = len(blocks)
        arr = (C.c_void_p * (nb * nb))()
        for i in range(nb):
            for j in range(nb):
                b = blocks[i][j]
                arr[i * nb + j] = None if b is None else b.h
                if b is not None:
                    b.h = None
        _chk(lib().pe_api_solver_set_operator_block(self.h, nb, arr))

    def level_block(self, ctx, l, i, j):
        """copy of block (i, j) of level l's operator as a capi.Mat, None for a zero block"""
        out = capi.Mat(ctx)
        _chk(lib().pe_api_solver_level_block(self.h, l, i, j, C.byref(out.h)))
        return out if out.h else None


def timer(name):
    s = C.c_double()
    _chk(lib().pe_api_timer_get(name.encode(), C.byref(s)))
    return s.value
