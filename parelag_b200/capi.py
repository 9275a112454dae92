"""ctypes binding of the C ABI declared in include/parelag_b200.h.

This is the reference-side binding stub a maintainer would write (see
INTEGRATION.md); the tests and bench.py drive the CUDA path through it.  There is
no CPU fallback: creating a context without a CUDA device raises.
"""
import ctypes as C
import os
import re

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libparelag_b200.so")
HEADER_PATHS = [os.path.join(os.path.dirname(_HERE), "include", "parelag_b200_local.h"),
                os.path.join(os.path.dirname(_HERE), "include", "parelag_b200.h"),
                os.path.join(os.path.dirname(_HERE), "include", "parelag_b200_api.h")]

_lib = None


class PEError(RuntimeError):
    pass


class ParCSRHost(C.Structure):
    """Mirror of struct pe_parcsr_host."""
    _fields_ = [
        ("global_num_rows", C.c_int64), ("global_num_cols", C.c_int64),
        ("first_row_index", C.c_int64), ("first_col_diag", C.c_int64),
        ("num_rows", C.c_int32), ("num_cols_diag", C.c_int32), ("num_cols_offd", C.c_int32),
        ("diag_i", C.c_void_p), ("diag_j", C.c_void_p), ("diag_data", C.c_void_p),
        ("offd_i", C.c_void_p), ("offd_j", C.c_void_p), ("offd_data", C.c_void_p),
        ("col_map_offd", C.c_void_p),
        ("num_sends", C.c_int32),
        ("send_procs", C.c_void_p), ("send_map_starts", C.c_void_p), ("send_map_elmts", C.c_void_p),
        ("num_recvs", C.c_int32),
        ("recv_procs", C.c_void_p), ("recv_vec_starts", C.c_void_p),
    ]


def declared_symbols():
    """Every function name declared in include/*.h (used by the CPU export test)."""
    names = []
    for path in HEADER_PATHS:
        if not os.path.exists(path):
            continue
        text = open(path).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names += re.findall(r"\b(pe_[a-z0-9_]+)\s*\(", text)
    return sorted(set(names))


def lib():
    """Load the shared library (raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PEError("%s not found: run `make` (or __graft_entry__.build())" % LIB_PATH)
        _lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        _lib.pe_last_error.restype = C.c_char_p
        _lib.pe_vec_size.restype = C.c_int64
        _lib.pe_ctx_launch_count.restype = C.c_int64
        _lib.pe_vec_device_ptr.restype = C.c_void_p
    return _lib


def _chk(rc):
    if rc != 0:
        raise PEError(lib().pe_last_error().decode())


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _i32(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.int32)


def _f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


class Ctx:
    def __init__(self, rank=0, nranks=1, device=0, nccl_id=None):
        self.h = C.c_void_p()
        _chk(lib().pe_ctx_create(rank, nranks, device, nccl_id, C.byref(self.h)))

    def sync(self):
        _chk(lib().pe_ctx_sync(self.h))

    def launch_count(self):
        return lib().pe_ctx_launch_count(self.h)

    def timer_start(self):
        _chk(lib().pe_ctx_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float()
        _chk(lib().pe_ctx_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def profile(self, enable):
        _chk(lib().pe_ctx_profile(self.h, 1 if enable else 0))

    def profile_get(self, kernel_id):
        cnt, ms, by = C.c_int64(), C.c_double(), C.c_double()
        _chk(lib().pe_ctx_profile_get(self.h, kernel_id, C.byref(cnt), C.byref(ms), C.byref(by)))
        return cnt.value, ms.value, by.value

    def flush_l2(self):
        _chk(lib().pe_ctx_flush_l2(self.h))

    def graph_begin(self):
        _chk(lib().pe_graph_begin(self.h))

    def graph_end(self):
        g = C.c_void_p()
        _chk(lib().pe_graph_end(self.h, C.byref(g)))
        return g

    def graph_launch(self, g):
        _chk(lib().pe_graph_launch(self.h, g))

    def close(self):
        if self.h:
            lib().pe_ctx_destroy(self.h)
            self.h = None


TUNE_SELL_MIN_ROWS = 0
TUNE_SELL_GROUP = 1
TUNE_PDL = 2
TUNE_GATHER_KEEP_PCT = 3
TUNE_P2P_HALO = 4
TUNE_FUSED_GS_MAX_MB = 5
TUNE_GS_SLABS = 6
TUNE_LOCAL_SMEM_BYTES = 7


def set_tuning(key, value):
    _chk(lib().pe_set_tuning(key, int(value)))


def get_tuning(key):
    return lib().pe_get_tuning(key)


# pe_api_solver_replay_mode values (include/parelag_b200_api.h): how the last preconditioner-mode V-cycle ran
REPLAY_DIRECT = 0
REPLAY_GRAPH = 1
REPLAY_PROGRAM = 2
REPLAY_MODE_NAMES = {REPLAY_DIRECT: "direct", REPLAY_GRAPH: "graph", REPLAY_PROGRAM: "program"}

# slots of pe_variant_counts (include/parelag_b200.h)
VARIANT_SLOTS = ("SPMV_SELL", "SPMV_STREAM", "SPMV_VECTOR",
                 "SPGEMM_SYM_T128", "SPGEMM_SYM_T1024", "SPGEMM_SYM_T8192", "SPGEMM_SYM_GMEM",
                 "SPGEMM_NUM_T128", "SPGEMM_NUM_T1024", "SPGEMM_NUM_T8192", "SPGEMM_NUM_GMEM",
                 "RELAX_TPR_1", "RELAX_TPR_2", "RELAX_TPR_4", "RELAX_TPR_8", "RELAX_TPR_16", "RELAX_TPR_32",
                 "TRACES_SMEM", "TRACES_GMEM", "EXT_SMEM", "EXT_GMEM",
                 "EXT_SPLIT_SMEM", "TRACES_GMEM_REUSE", "EXT_GMEM_REUSE", "SPMV_SELL_SIGNS",
                 "SELL_GS_G4_SINGLE", "SELL_GS_G4_PIPE", "SELL_GS_G8_SINGLE", "SELL_GS_G8_PIPE",
                 "SELL_GS_G12_SINGLE", "SELL_GS_G12_PIPE",
                 "SELL_SPMV_G4_SINGLE", "SELL_SPMV_G4_PIPE", "SELL_SPMV_G8_SINGLE", "SELL_SPMV_G8_PIPE",
                 "SELL_SPMV_G12_SINGLE", "SELL_SPMV_G12_PIPE")
(SPMV_SELL, SPMV_STREAM, SPMV_VECTOR,
 SPGEMM_SYM_T128, SPGEMM_SYM_T1024, SPGEMM_SYM_T8192, SPGEMM_SYM_GMEM,
 SPGEMM_NUM_T128, SPGEMM_NUM_T1024, SPGEMM_NUM_T8192, SPGEMM_NUM_GMEM,
 RELAX_TPR_1, RELAX_TPR_2, RELAX_TPR_4, RELAX_TPR_8, RELAX_TPR_16, RELAX_TPR_32,
 TRACES_SMEM, TRACES_GMEM, EXT_SMEM, EXT_GMEM,
 EXT_SPLIT_SMEM, TRACES_GMEM_REUSE, EXT_GMEM_REUSE, SPMV_SELL_SIGNS,
 SELL_GS_G4_SINGLE, SELL_GS_G4_PIPE, SELL_GS_G8_SINGLE, SELL_GS_G8_PIPE, SELL_GS_G12_SINGLE, SELL_GS_G12_PIPE,
 SELL_SPMV_G4_SINGLE, SELL_SPMV_G4_PIPE, SELL_SPMV_G8_SINGLE, SELL_SPMV_G8_PIPE, SELL_SPMV_G12_SINGLE,
 SELL_SPMV_G12_PIPE) = range(len(VARIANT_SLOTS))


def sell_group_slot(kernel, G, single):
    """slot of the (G, single) entry-group variant of k_sell_gs (kernel "gs") or k_sell_spmv ("spmv")"""
    base = SELL_GS_G4_SINGLE if kernel == "gs" else SELL_SPMV_G4_SINGLE
    return base + 2 * (G // 4 - 1) + (0 if single else 1)


def variant_counts(reset=False):
    """Rows / agglomerates each size-dispatched kernel variant was given since the last reset (process-wide):
    int64 array indexed by the slot constants above.  reset: zero the counters after reading them."""
    out = np.zeros(len(VARIANT_SLOTS), dtype=np.int64)
    _chk(lib().pe_variant_counts(_ptr(out), len(VARIANT_SLOTS), 1 if reset else 0))
    return out


def nccl_unique_id():
    buf = C.create_string_buffer(128)
    _chk(lib().pe_nccl_get_unique_id(buf))
    return buf.raw


class Vec:
    def __init__(self, ctx, n=None, data=None):
        self.ctx = ctx
        if data is not None:
            data = _f64(data)
            n = data.size
        self.n = int(n)
        self.h = C.c_void_p()
        _chk(lib().pe_vec_create(ctx.h, C.c_int64(self.n), C.byref(self.h)))
        if data is not None:
            self.upload(data)

    def upload(self, data):
        data = _f64(data)
        assert data.size == self.n
        _chk(lib().pe_vec_upload(self.h, _ptr(data)))

    def download(self):
        out = np.empty(self.n, dtype=np.float64)
        _chk(lib().pe_vec_download(self.h, _ptr(out)))
        return out

    def fill(self, v):
        _chk(lib().pe_vec_fill(self.h, C.c_double(v)))

    def copy_from(self, src):
        _chk(lib().pe_vec_copy(src.h, self.h))

    def axpby(self, a, x, b):
        """self = a*x + b*self"""
        _chk(lib().pe_vec_axpby(C.c_double(a), x.h, C.c_double(b), self.h))

    def dot(self, other):
        out = C.c_double()
        _chk(lib().pe_vec_dot(self.h, other.h, C.byref(out)))
        return out.value

    def free(self):
        if self.h:
            lib().pe_vec_free(self.h)
            self.h = None


class Mat:
    """Device ParCSR matrix.  Build from a scipy CSR (single rank) or from the raw
    diag/offd/comm-package arrays of a hypre ParCSR matrix."""

    def __init__(self, ctx, handle=None):
        self.ctx = ctx
        self.h = handle if handle is not None else C.c_void_p()

    @staticmethod
    def from_scipy(ctx, A):
        A = A.tocsr()
        return Mat.from_parcsr(ctx, A.shape[0], A.shape[1], A.indptr, A.indices, A.data)

    @staticmethod
    def from_parcsr(ctx, num_rows, num_cols_diag, diag_i, diag_j, diag_data,
                    offd_i=None, offd_j=None, offd_data=None, col_map_offd=None,
                    global_num_rows=None, global_num_cols=None, first_row=0, first_col=0,
                    send_procs=None, send_map_starts=None, send_map_elmts=None,
                    recv_procs=None, recv_vec_starts=None):
        keep = [_i32(diag_i), _i32(diag_j), _f64(diag_data), _i32(offd_i), _i32(offd_j),
                _f64(offd_data),
                None if col_map_offd is None else np.ascontiguousarray(col_map_offd, dtype=np.int64),
                _i32(send_procs), _i32(send_map_starts), _i32(send_map_elmts),
                _i32(recv_procs), _i32(recv_vec_starts)]
        H = ParCSRHost()
        H.global_num_rows = num_rows if global_num_rows is None else global_num_rows
        H.global_num_cols = num_cols_diag if global_num_cols is None else global_num_cols
        H.first_row_index = first_row
        H.first_col_diag = first_col
        H.num_rows = num_rows
        H.num_cols_diag = num_cols_diag
        H.num_cols_offd = 0 if col_map_offd is None else len(col_map_offd)
        (H.diag_i, H.diag_j, H.diag_data, H.offd_i, H.offd_j, H.offd_data, H.col_map_offd,
         H.send_procs, H.send_map_starts, H.send_map_elmts, H.recv_procs,
         H.recv_vec_starts) = [_ptr(a) for a in keep]
        H.num_sends = 0 if send_procs is None else len(send_procs)
        H.num_recvs = 0 if recv_procs is None else len(recv_procs)
        m = Mat(ctx)
        _chk(lib().pe_mat_upload(ctx.h, C.byref(H), C.byref(m.h)))
        return m

    def info(self):
        nr, ncd, nco = C.c_int32(), C.c_int32(), C.c_int32()
        nd, no = C.c_int64(), C.c_int64()
        _chk(lib().pe_mat_info(self.h, C.byref(nr), C.byref(ncd), C.byref(nco), C.byref(nd),
                               C.byref(no)))
        return nr.value, ncd.value, nco.value, nd.value, no.value

    def to_scipy(self):
        """Download the diag block as scipy CSR (single-rank matrices)."""
        import scipy.sparse as sp
        nr, ncd, nco, nd, no = self.info()
        I = np.empty(nr + 1, dtype=np.int32)
        J = np.empty(nd, dtype=np.int32)
        A = np.empty(nd, dtype=np.float64)
        _chk(lib().pe_mat_download(self.h, _ptr(I), _ptr(J), _ptr(A), None, None, None, None))
        return sp.csr_matrix((A, J, I), shape=(nr, ncd))

    def download_parcsr(self):
        """All blocks of a (distributed) ParCSR matrix: dict as parelag_b200.par.OwnedParCSR.arrays()."""
        nr, ncd, nco, nd, no = self.info()
        gr, gc, fr, fc = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
        _chk(lib().pe_mat_global_info(self.h, C.byref(gr), C.byref(gc), C.byref(fr), C.byref(fc)))
        d = dict(first_row=fr.value, first_col=fc.value, nrows=nr, ncols_diag=ncd, global_rows=gr.value, global_cols=gc.value,
                 diag_i=np.empty(nr + 1, dtype=np.int32), diag_j=np.empty(nd, dtype=np.int32), diag_a=np.empty(nd),
                 offd_i=np.zeros(nr + 1, dtype=np.int32), offd_j=np.empty(no, dtype=np.int32), offd_a=np.empty(no),
                 col_map_offd=np.empty(nco, dtype=np.int64))
        _chk(lib().pe_mat_download(self.h, _ptr(d["diag_i"]), _ptr(d["diag_j"]), _ptr(d["diag_a"]), _ptr(d["offd_i"]),
                                   _ptr(d["offd_j"]) if no else None, _ptr(d["offd_a"]) if no else None,
                                   _ptr(d["col_map_offd"]) if nco else None))
        return d

    def transpose(self):
        out = Mat(self.ctx)
        _chk(lib().pe_mat_transpose(self.ctx.h, self.h, C.byref(out.h)))
        return out

    def spmv(self, x, y, alpha=1.0, beta=0.0):
        _chk(lib().pe_spmv(self.ctx.h, C.c_double(alpha), self.h, x.h, C.c_double(beta), y.h))

    def spmv_t(self, x, y, alpha=1.0, beta=0.0):
        _chk(lib().pe_spmv_t(self.ctx.h, C.c_double(alpha), self.h, x.h, C.c_double(beta), y.h))

    def residual(self, x, b, r):
        _chk(lib().pe_residual(self.ctx.h, self.h, x.h, b.h, r.h))

    def fix_zero_rows(self):
        n = C.c_int32()
        _chk(lib().pe_fix_zero_rows(self.ctx.h, self.h, C.byref(n)))
        return n.value

    # ---- src/hypreExtension utilities
    def delete_zeros(self, tol):
        _chk(lib().pe_mat_delete_zeros(self.ctx.h, self.h, C.c_double(tol)))

    def sign(self, tol=1e-9):
        _chk(lib().pe_mat_sign(self.ctx.h, self.h, C.c_double(tol)))

    def norms(self):
        out = np.zeros(4)
        _chk(lib().pe_mat_norms(self.ctx.h, self.h, _ptr(out)))
        return dict(l1=out[0], linf=out[1], max=out[2], fro=out[3])

    def compare(self, other, tol):
        f = C.c_int32()
        _chk(lib().pe_mat_compare(self.ctx.h, self.h, other.h, C.c_double(tol), C.byref(f)))
        return f.value

    @staticmethod
    def diagonal(ctx, n, d=None):
        out = Mat(ctx)
        _chk(lib().pe_mat_diagonal(ctx.h, n, None if d is None else d.h, C.byref(out.h)))
        return out

    def free(self):
        if self.h:
            lib().pe_mat_free(self.h)
            self.h = None


def rdp(ctx, R, d, P):
    out = Mat(ctx)
    _chk(lib().pe_rdp(ctx.h, R.h, d.h, P.h, C.byref(out.h)))
    return out


def spgemm(ctx, A, B):
    out = Mat(ctx)
    _chk(lib().pe_spgemm(ctx.h, A.h, B.h, C.byref(out.h)))
    return out


def rap(ctx, A, P, R=None):
    out = Mat(ctx)
    _chk(lib().pe_rap(ctx.h, None if R is None else R.h, A.h, P.h, C.byref(out.h)))
    return out


def spadd(ctx, a, A, b, B):
    out = Mat(ctx)
    _chk(lib().pe_spadd(ctx.h, C.c_double(a), A.h, C.c_double(b), B.h, C.byref(out.h)))
    return out


SMOOTHER_TYPES = {"Jacobi": 0, "L1 Jacobi": 1, "L1 Gauss-Seidel": 2, "L1 Gauss-Seidel Truncated": 4,
                  "Lumped Jacobi": 5, "Gauss-Seidel": 6, "Chebyshev": 16}
GS_NATURAL, GS_MULTICOLOR = 0, 1


class Smoother:
    def __init__(self, ctx, A, type=2, sweeps=1, damping=1.0, omega=1.0, cheby_order=2,
                 cheby_fraction=0.3, ordering=GS_NATURAL):
        self.ctx, self.A = ctx, A
        self.h = C.c_void_p()
        _chk(lib().pe_smoother_create(ctx.h, A.h, type, sweeps, C.c_double(damping),
                                      C.c_double(omega), cheby_order, C.c_double(cheby_fraction),
                                      ordering, C.byref(self.h)))

    def apply(self, b, x, iterative_mode=True):
        _chk(lib().pe_smoother_apply(self.h, b.h, x.h, 1 if iterative_mode else 0))

    def l1(self):
        n = self.A.info()[0]
        out = np.empty(n)
        _chk(lib().pe_smoother_get_l1(self.h, _ptr(out)))
        return out

    def order(self):
        n = self.A.info()[0]
        ns = C.c_int32()
        _chk(lib().pe_smoother_get_order(self.h, None, C.byref(ns), None))
        order = np.empty(n, dtype=np.int32)
        starts = np.empty(ns.value + 1, dtype=np.int32)
        _chk(lib().pe_smoother_get_order(self.h, _ptr(order), C.byref(ns), _ptr(starts)))
        return order, starts

    def eig(self):
        a, b = C.c_double(), C.c_double()
        _chk(lib().pe_smoother_get_eig(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def free(self):
        if self.h:
            lib().pe_smoother_free(self.h)
            self.h = None
