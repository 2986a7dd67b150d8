"""ctypes binding of ``libsmcp_b200.so`` and the product backend of the drivers.

PyTorch-free: NumPy for host buffers, ctypes for the C ABI declared in
``include/smcp_b200.h``.  There is no CPU fallback — if the shared library is missing or no
CUDA device is present, constructing a ``DeviceBackend`` raises ``RuntimeError``.
"""
from __future__ import annotations

import ctypes as C
import os
import numpy as np

from .symbolic import task_partition

_LIB = None
_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libsmcp_b200.so")

_i64p = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_i8p = np.ctypeslib.ndpointer(dtype=np.int8, flags="C_CONTIGUOUS")


class SymDesc(C.Structure):
    _fields_ = [(k, C.c_int64) for k in ("n", "nsn", "nvp", "nblk", "nupd")] + \
               [(k, C.c_void_p) for k in ("snptr", "snpar", "rowptr", "rowidx", "blkptr", "updptr", "chptr",
                                          "chidx", "relptr", "relidx", "aaidx", "vec2blk", "diagblk", "wdot")] + \
               [("ntask", C.c_int64)] + \
               [(k, C.c_void_p) for k in ("task_ptr", "task_sn", "dep_ptr", "dep_idx")]


# every symbol declared in include/smcp_b200.h: name -> (restype, argtypes)
_vp, _dp, _i64, _int, _dbl = C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_double
API = {
    "smcp_ctx_create": (_int, [_int, C.POINTER(_vp)]),
    "smcp_ctx_destroy": (_int, [_vp]),
    "smcp_ctx_sync": (_int, [_vp]),
    "smcp_last_error": (C.c_char_p, []),
    "smcp_version": (_int, []),
    "smcp_ctx_launch_count": (_i64, [_vp]),
    "smcp_timer_start": (_int, [_vp]),
    "smcp_timer_stop": (_int, [_vp, C.POINTER(_dbl)]),
    "smcp_prof_enable": (_int, [_vp, _int]),
    "smcp_prof_get": (_int, [_vp, C.c_char_p, C.POINTER(_dbl), C.POINTER(_i64)]),
    "smcp_prof_get_work": (_int, [_vp, C.c_char_p, C.POINTER(_dbl)]),
    "smcp_prof_list": (_int, [_vp, C.c_char_p, _i64]),
    "smcp_prof_reset": (_int, [_vp]),
    "smcp_region_get": (_int, [_vp, C.c_char_p, C.POINTER(_dbl), C.POINTER(_i64)]),
    "smcp_region_reset": (_int, [_vp]),
    "smcp_region_list": (_int, [_vp, C.c_char_p, _i64]),
    "smcp_flush_l2": (_int, [_vp]),
    "smcp_sym_create": (_int, [_vp, C.POINTER(SymDesc), C.POINTER(_vp)]),
    "smcp_sym_destroy": (_int, [_vp]),
    "smcp_sym_reserve": (_int, [_vp, _i64]),
    "smcp_csp_alloc": (_int, [_vp, _i64, C.POINTER(_dp)]),
    "smcp_csp_free": (_int, [_vp, _dp]),
    "smcp_csp_copy": (_int, [_vp, _dp, _dp, _i64]),
    "smcp_csp_from_vec": (_int, [_vp, _dp, _f64p]),
    "smcp_csp_to_vec": (_int, [_vp, _dp, _f64p]),
    "smcp_csp_get": (_int, [_vp, _dp, _f64p]),
    "smcp_csp_set": (_int, [_vp, _dp, _f64p]),
    "smcp_csp_axpy": (_int, [_vp, _dbl, _dp, _dp]),
    "smcp_csp_scal": (_int, [_vp, _dbl, _dp]),
    "smcp_csp_dot": (_int, [_vp, _dp, _dp, C.POINTER(_dbl)]),
    "smcp_csp_sumlogdiag": (_int, [_vp, _dp, C.POINTER(_dbl)]),
    "smcp_csp_cholesky": (_int, [_vp, _dp, _i64, _i32p]),
    "smcp_csp_completion": (_int, [_vp, _dp, _i64, _i32p]),
    "smcp_csp_projected_inverse": (_int, [_vp, _dp, _i64]),
    "smcp_csp_llt": (_int, [_vp, _dp, _i64]),
    "smcp_csp_probe": (_int, [_vp, _int, _dp, _dp, _f64p, _i64, _i32p, _f64p]),
    "smcp_csp_trsm": (_int, [_vp, _dp, _dp, _i64, _i64, _int]),
    "smcp_csp_sample": (_int, [_vp, _dp, C.c_uint64, _i64, _dp, _i64, _i64]),
    "smcp_round_pm1": (_int, [_vp, _dp, C.c_uint64, _i64, _i64, _i64, _i64p, _i64p, _f64p, _f64p,
                              np.ctypeslib.ndpointer(dtype=np.int8, flags="C_CONTIGUOUS"), C.POINTER(_i64)]),
    "smcp_round_pm1_ls": (_int, [_vp, _dp, C.c_uint64, _i64, _i64, _i64, _i64p, _i64p, _f64p, _i64, _dbl, _f64p, _f64p,
                                 _i8p, C.POINTER(_i64), _i64p]),
    "smcp_pm1_local_search": (_int, [_vp, _i64, _i64, _i8p, _i64, _i64p, _i64p, _f64p, _i64, _dbl, _f64p, _i64p]),
    "smcp_round_pm1_tabu": (_int, [_vp, _dp, C.c_uint64, _i64, _i64, _i64, _i64p, _i64p, _f64p, _i64, _dbl, _f64p, _f64p,
                                   _i8p, C.POINTER(_i64), _i64p, _i64, _i64, _f64p, _i64p, _i64p]),
    "smcp_pm1_tabu_search": (_int, [_vp, _i64, _i64, _i8p, _i64, _i64p, _i64p, _f64p, _i64, _i64, _f64p, _i64p, _i64p]),
    "smcp_lowrank_solve": (_int, [_vp, _i64, _i64, _i64, _i64p, _i64p, _f64p, _f64p, C.c_uint64, _i64, _dbl, _f64p, _f64p,
                                  _f64p, C.POINTER(_i64), C.POINTER(_i64)]),
    "smcp_round_pm1_factor": (_int, [_vp, _i64, _i64, _f64p, C.c_uint64, _i64, _i64, _i64, _i64p, _i64p, _f64p, _i64, _dbl,
                                     _i64, _i64, _vp, _vp, _f64p, _i8p, C.POINTER(_i64), _vp, _vp, _vp]),
    "smcp_hess_create": (_int, [_vp, _dp, _dp, C.POINTER(_vp)]),
    "smcp_hess_destroy": (_int, [_vp]),
    "smcp_hess_apply": (_int, [_vp, _dp, _i64, _int]),
    "smcp_hess_apply_half": (_int, [_vp, _dp, _i64, _int, _int]),
    "smcp_op_create": (_int, [_vp, _i64, _i64, _i64p, _i64p, _f64p, C.POINTER(_vp)]),
    "smcp_op_destroy": (_int, [_vp]),
    "smcp_op_set_entry_coords": (_int, [_vp, _i64p, _i64p]),
    "smcp_op_dense_rows": (_int, [_vp, C.POINTER(_i64)]),
    "smcp_op_amap": (_int, [_vp, _dp, _i64, _f64p]),
    "smcp_op_aadj": (_int, [_vp, _f64p, _dp]),
    "smcp_kkt_assemble": (_int, [_vp, _vp, _i64, _i64]),
    "smcp_kkt_assemble_cyclic": (_int, [_vp, _vp, _i64, _int, _int]),
    "smcp_kkt_assemble_syrk": (_int, [_vp, _vp]),
    "smcp_kkt_z_tmul": (_int, [_vp, _dp, _f64p]),
    "smcp_kkt_z_mul": (_int, [_vp, _f64p, _dp]),
    "smcp_kkt_factor_qr": (_int, [_vp, _vp, _i32p]),
    "smcp_kkt_qr_solve": (_int, [_vp, _dp, _f64p, _f64p, _dp]),
    "smcp_kkt_factor": (_int, [_vp, _i32p]),
    "smcp_kkt_factor_dist": (_int, [_vp, _int, _int, _i32p]),
    "smcp_kkt_factor_block": (_int, [_vp, _i64, _int, _int, _i32p]),
    "smcp_dense_potrf": (_int, [_vp, _f64p, _i64, _i64, _i64, _i32p, C.POINTER(_dbl)]),
    "smcp_dense_trsm": (_int, [_vp, _int, _f64p, _i64, _i64, _f64p, _i64, _i64, C.POINTER(_dbl)]),
    "smcp_dense_gemm": (_int, [_vp, _int, _int, _f64p, _i64, _f64p, _i64, _f64p, _i64, _i64, _i64, _i64, _dbl, _int, _int,
                               C.POINTER(_dbl)]),
    "smcp_dense_geqrf": (_int, [_vp, _f64p, _i64, _i64, _i64, _f64p, C.POINTER(_dbl)]),
    "smcp_dense_orgqr": (_int, [_vp, _f64p, _i64, _i64, _i64, _f64p, C.POINTER(_dbl)]),
    "smcp_kkt_solve": (_int, [_vp, _f64p]),
    "smcp_kkt_get_H": (_int, [_vp, _f64p]),
    "smcp_kkt_set_H": (_int, [_vp, _f64p]),
    "smcp_kkt_H_devptr": (_int, [_vp, C.POINTER(_dp)]),
    "smcp_comm_unique_id": (_int, [C.c_char_p]),
    "smcp_comm_init": (_int, [_vp, _int, _int, C.c_char_p]),
    "smcp_comm_destroy": (_int, [_vp]),
    "smcp_kkt_allgather": (_int, [_vp, _i64, _int, _int]),
    "smcp_host_min_degree": (_int, [_i64, _i64p, _i64p, _i64p]),
    "smcp_host_maxcardsearch": (_int, [_i64, _i64p, _i64p, _i64p]),
    "smcp_host_embed": (_int, [_i64, _i64p, _i64p, _i64p, C.c_void_p, C.c_void_p]),
    "smcp_host_aaidx": (_int, [_i64, _i64p, _i64p, _i64p, _i64p, _i64p, _i64p, _i64p, _i64p]),
    "smcp_host_supernodes": (_int, [_i64, _i64p, _i64p, C.POINTER(_i64), _i64p, _i64p, _i64p, _i64p, _i64p, _i64p, _i64p]),
}


def load_library(path=None):
    """Load the shared library and declare every entry point (raises if it is missing)."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    path = path or os.environ.get("SMCP_B200_LIB") or _LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(nvcc, sm_100a). There is no CPU fallback." % path)
    lib = C.CDLL(path)
    for name, (res, args) in API.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if os.environ.get("SMCP_B200_HOSTPROF"):
        lib = _HostProf(lib)
    _LIB = lib
    return lib


HOSTPROF = {}      # name -> [calls, seconds]: host wall time spent inside each C-ABI call


class _HostProf:
    """Debug aid (SMCP_B200_HOSTPROF=1): wraps every entry point with a host wall-clock counter so
    that a blocking call shows up by name; results in ``device.HOSTPROF``."""

    def __init__(self, lib):
        import time
        for name in API:
            fn = getattr(lib, name)

            def wrapped(*a, _fn=fn, _name=name, _t=time.perf_counter):
                t0 = _t()
                r = _fn(*a)
                e = HOSTPROF.setdefault(_name, [0, 0.0])
                e[0] += 1
                e[1] += _t() - t0
                return r
            setattr(self, name, wrapped)


class DeviceError(RuntimeError):
    pass


def _ck(lib, rc):
    if rc != 0:
        raise DeviceError("libsmcp_b200: %s" % lib.smcp_last_error().decode("utf-8", "replace"))


class Context:
    """One CUDA context/stream per process and GPU (``smcp_ctx``)."""
    _cache = {}

    def __init__(self, device=0):
        self.lib = load_library()
        h = C.c_void_p()
        _ck(self.lib, self.lib.smcp_ctx_create(int(device), C.byref(h)))
        self.h = h
        self.device = device

    @classmethod
    def get(cls, device=None):
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", os.environ.get("SMCP_DEVICE", "0")))
        if device not in cls._cache:
            cls._cache[device] = Context(device)
        return cls._cache[device]

    def sync(self):
        _ck(self.lib, self.lib.smcp_ctx_sync(self.h))

    def launch_count(self):
        return int(self.lib.smcp_ctx_launch_count(self.h))

    def timer_start(self):
        _ck(self.lib, self.lib.smcp_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_double()
        _ck(self.lib, self.lib.smcp_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def prof_enable(self, on=True):
        _ck(self.lib, self.lib.smcp_prof_enable(self.h, int(bool(on))))

    def prof_reset(self):
        _ck(self.lib, self.lib.smcp_prof_reset(self.h))

    def prof_get(self, name):
        ms, n = C.c_double(), C.c_int64()
        _ck(self.lib, self.lib.smcp_prof_get(self.h, name.encode(), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def prof_get_work(self, name):
        w = C.c_double()
        _ck(self.lib, self.lib.smcp_prof_get_work(self.h, name.encode(), C.byref(w)))
        return w.value

    def prof_names(self):
        buf = C.create_string_buffer(8192)
        _ck(self.lib, self.lib.smcp_prof_list(self.h, buf, 8192))
        s = buf.value.decode()
        return s.split(",") if s else []

    def region_get(self, name):
        ms, n = C.c_double(), C.c_int64()
        _ck(self.lib, self.lib.smcp_region_get(self.h, name.encode(), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def region_names(self):
        buf = C.create_string_buffer(8192)
        _ck(self.lib, self.lib.smcp_region_list(self.h, buf, 8192))
        s = buf.value.decode()
        return s.split(",") if s else []

    def region_reset(self):
        _ck(self.lib, self.lib.smcp_region_reset(self.h))

    def flush_l2(self):
        _ck(self.lib, self.lib.smcp_flush_l2(self.h))


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


_COMM = None          # (rank, nranks, block) once init_comm() has built the NCCL communicator
TRAFFIC = {"h2d": 0, "d2h": 0}     # host<->device bytes moved through the API (bench.py reads it)


def init_comm(rank, nranks, unique_id, block=64, device=None):
    """Create the library-owned NCCL communicator (one process per GPU).  ``unique_id`` is the
    128-byte id produced by ``comm_unique_id()`` on rank 0 and distributed by the launcher."""
    global _COMM
    ctx = Context.get(device)
    _ck(ctx.lib, ctx.lib.smcp_comm_init(ctx.h, int(rank), int(nranks), bytes(unique_id)))
    _COMM = (int(rank), int(nranks), int(block))


def comm_unique_id():
    lib = load_library()
    buf = C.create_string_buffer(128)
    _ck(lib, lib.smcp_comm_unique_id(buf))
    return buf.raw


def owned_column_blocks(m, rank, nranks, block):
    """1-D block-cyclic ownership of the columns of H: [(j0, j1), ...] for ``rank``."""
    return [(c0, min(m, c0 + block)) for c0 in range(rank * block, m, nranks * block)]


class DeviceBackend:
    """``BackendProtocol`` (see ``smcp_b200.chordal``) on the CUDA library."""
    name = "cuda-sm100a"
    batched_probes = True        # line-search probes are evaluated as one device batch

    def __init__(self, symb, device=None, small_work=200000, comm=None):
        self.ctx = Context.get(device)
        self.lib = lib = self.ctx.lib
        self.symb = symb
        self.comm = comm if comm is not None else _COMM      # (rank, nranks, block)
        tp, ts, dp, di, _ = task_partition(symb, small_work)
        keep = dict(snptr=_i64(symb.snptr), snpar=_i64(symb.snpar), rowptr=_i64(symb.rowptr),
                    rowidx=_i64(symb.rowidx), blkptr=_i64(symb.blkptr), updptr=_i64(symb.updptr),
                    chptr=_i64(symb.chptr), chidx=_i64(symb.chidx), relptr=_i64(symb.relptr),
                    relidx=_i64(symb.relidx), aaidx=_i64(symb.aaidx), vec2blk=_i64(symb.vec2blk),
                    diagblk=_i64(symb.diag_blk), wdot=np.ascontiguousarray(symb.wdot, dtype=np.float64),
                    task_ptr=_i64(tp), task_sn=_i64(ts), dep_ptr=_i64(dp), dep_idx=_i64(di))
        d = SymDesc()
        d.n, d.nsn, d.nvp, d.nblk, d.nupd = symb.n, symb.nsn, symb.nvp, symb.nblk, symb.nupd
        d.ntask = len(tp) - 1
        for k, v in keep.items():
            setattr(d, k, v.ctypes.data if v.size else None)
        h = C.c_void_p()
        _ck(lib, lib.smcp_sym_create(self.ctx.h, C.byref(d), C.byref(h)))
        self.sym = h
        # patterns with large frontal matrices: single-matrix operations go to the dense multi-CTA
        # path (csrc/bigfront.cu), so the 8 probes of a bisection run one after the other through
        # it instead of as one 255-candidate batch through the CTA-per-supernode kernels
        # (same rule as big_setup in csrc/bigfront.cu)
        nj = np.diff(symb.rowptr).astype(np.float64)
        nn = np.diff(symb.snptr).astype(np.float64)
        na = nj - nn
        fl = 4.0 * nn ** 3 + 6.0 * na * nn ** 2 + 6.0 * na ** 2 * nn
        thr_flops = float(os.environ.get("SMCP_B200_BIG_FLOPS", "2e6"))
        thr_nj = int(os.environ.get("SMCP_B200_BIG_NJ", "0"))
        thr_compl = float(os.environ.get("SMCP_B200_BIG_COMPL_FLOPS", "6e5" if thr_flops > 0 else "0"))   # = bigfront.cu
        has_big = symb.nsn > 0 and ((thr_flops > 0 and fl.max() >= thr_flops) or (thr_nj > 0 and nj.max() >= thr_nj)
                                    or (thr_flops > 0 and thr_compl > 0 and (na ** 3).max() / 3.0 >= thr_compl))
        self.batched_probes = not (has_big and (nj.max() > 8 or thr_nj > 0))
        if self.batched_probes and symb.nblk * 255 * 8 <= (1 << 30):
            # workspaces of the batched line-search probes (255 candidates) sized at setup time
            _ck(lib, lib.smcp_sym_reserve(h, 255))
        elif self.batched_probes:
            # 255 candidate matrices would not fit the workspace budget: the 8 probes of a bisection run one
            # after the other (no allocation inside the iterations, no out-of-memory surprise)
            self.batched_probes = False
        self._pool = []
        # chordal-matrix buffers are recycled through this pool; fill it up front so that no
        # cudaMalloc (a synchronising driver call) happens inside the IPM iterations
        # (up to 40 buffers within 8 GB: rand_SDP n = 2000 has 12 MB per matrix; without the pool the first iterations
        # with extra centering steps stalled 70-120 ms each in cudaMalloc, gpurun_out/r02_v36_C3.log)
        nprefill = int(min(40, (8 << 30) // max(1, symb.nblk * 8)))
        for _ in range(nprefill):
            p = C.c_void_p()
            _ck(lib, lib.smcp_csp_alloc(h, 1, C.byref(p)))
            self._pool.append(p)
        self._op = None
        self._tok = None
        self.m = 0
        self.Ns = 0

    def __del__(self):
        try:
            if self._tok is not None:
                self.lib.smcp_hess_destroy(self._tok)
            if self._op is not None:
                self.lib.smcp_op_destroy(self._op)
            for p in self._pool:
                self.lib.smcp_csp_free(self.sym, p)
            self.lib.smcp_sym_destroy(self.sym)
        except Exception:
            pass

    # -- storage ----------------------------------------------------------------------
    def _alloc(self, zero):
        if self._pool:
            p = self._pool.pop()
            if zero:
                _ck(self.lib, self.lib.smcp_csp_scal(self.sym, 0.0, p))
            return p
        p = C.c_void_p()
        _ck(self.lib, self.lib.smcp_csp_alloc(self.sym, 1, C.byref(p)))
        return p

    def new(self):
        return self._alloc(True)

    def release(self, buf):
        if buf is not None and len(self._pool) < 64:
            self._pool.append(buf)
        elif buf is not None:
            self.lib.smcp_csp_free(self.sym, buf)

    def clone(self, buf):
        p = self._alloc(False)
        _ck(self.lib, self.lib.smcp_csp_copy(self.sym, p, buf, 1))
        return p

    def from_vec(self, v):
        TRAFFIC["h2d"] += 8 * self.symb.nvp
        p = self._alloc(False)
        _ck(self.lib, self.lib.smcp_csp_from_vec(self.sym, p, np.ascontiguousarray(v, dtype=np.float64)))
        return p

    def to_vec(self, buf):
        TRAFFIC["d2h"] += 8 * self.symb.nvp
        out = np.empty(self.symb.nvp)
        _ck(self.lib, self.lib.smcp_csp_to_vec(self.sym, buf, out))
        return out

    def get_blk(self, buf):
        out = np.empty(self.symb.nblk)
        _ck(self.lib, self.lib.smcp_csp_get(self.sym, buf, out))
        return out

    def set_blk(self, host):
        p = self._alloc(False)
        _ck(self.lib, self.lib.smcp_csp_set(self.sym, p, np.ascontiguousarray(host, dtype=np.float64)))
        return p

    # -- level 1 ----------------------------------------------------------------------
    def axpy(self, a, x, y):
        _ck(self.lib, self.lib.smcp_csp_axpy(self.sym, float(a), x, y))

    def scal(self, a, x):
        _ck(self.lib, self.lib.smcp_csp_scal(self.sym, float(a), x))

    def dot(self, x, y):
        TRAFFIC["d2h"] += 8
        out = C.c_double()
        _ck(self.lib, self.lib.smcp_csp_dot(self.sym, x, y, C.byref(out)))
        return out.value

    def sumlogdiag(self, buf):
        out = C.c_double()
        _ck(self.lib, self.lib.smcp_csp_sumlogdiag(self.sym, buf, C.byref(out)))
        return out.value

    # -- factorizations ---------------------------------------------------------------
    def cholesky(self, buf):
        info = np.zeros(1, dtype=np.int32)
        _ck(self.lib, self.lib.smcp_csp_cholesky(self.sym, buf, 1, info))
        if info[0]:
            raise ArithmeticError("matrix is not positive definite")

    def completion(self, buf):
        info = np.zeros(1, dtype=np.int32)
        _ck(self.lib, self.lib.smcp_csp_completion(self.sym, buf, 1, info))
        if info[0]:
            raise ArithmeticError("matrix has no positive definite completion")

    def projected_inverse(self, buf):
        _ck(self.lib, self.lib.smcp_csp_projected_inverse(self.sym, buf, 1))

    def llt(self, buf):
        _ck(self.lib, self.lib.smcp_csp_llt(self.sym, buf, 1))

    def probe(self, kind, x, dx, gammas):
        """Batched step-length probes: verdicts (True = in cone) and sum(log(diag(L)))."""
        g = np.ascontiguousarray(gammas, dtype=np.float64)
        info = np.zeros(len(g), dtype=np.int32)
        sld = np.zeros(len(g))
        _ck(self.lib, self.lib.smcp_csp_probe(self.sym, 0 if kind == "cholesky" else 1, x, dx, g, len(g), info, sld))
        return info == 0, sld

    # -- contiguous batches (layout of the Schur assembly and the probes) ----------------
    def alloc_batch(self, count):
        p = C.c_void_p()
        _ck(self.lib, self.lib.smcp_csp_alloc(self.sym, int(count), C.byref(p)))
        return p

    def free_batch(self, buf):
        _ck(self.lib, self.lib.smcp_csp_free(self.sym, buf))

    def _slot(self, buf, k):
        return C.c_void_p(buf.value + 8 * k * self.symb.nblk)

    def set_batch(self, buf, host):
        host = np.ascontiguousarray(host, dtype=np.float64)
        for k in range(host.shape[0]):
            _ck(self.lib, self.lib.smcp_csp_set(self.sym, self._slot(buf, k), host[k]))

    def get_batch(self, buf, count):
        out = np.empty((count, self.symb.nblk))
        for k in range(count):
            _ck(self.lib, self.lib.smcp_csp_get(self.sym, self._slot(buf, k), out[k]))
        return out

    def trsm(self, Lbuf, B, trans="N"):
        """``chompack.trsm(L, B[, trans='T'])`` (``solvers.py:491-492``): B <- L^{-1} B or L^{-T} B for a
        dense n x k matrix whose rows are in the internal order of ``symb``.  Returns a new array
        (the device path keeps such blocks resident; this host round trip exists for tests)."""
        B = np.asarray(B, dtype=np.float64)
        n, k = B.shape
        nblk = self.symb.nblk
        count = max(1, -(-(n * k) // nblk))
        flat = np.zeros(count * nblk)
        flat[:n * k] = B.reshape(-1, order="F")
        buf = self.alloc_batch(count)
        try:
            self.set_batch(buf, flat.reshape(count, nblk))
            _ck(self.lib, self.lib.smcp_csp_trsm(self.sym, Lbuf, buf, n, k, 1 if trans == "T" else 0))
            out = self.get_batch(buf, count).reshape(-1)[:n * k].reshape(n, k, order="F")
        finally:
            self.free_batch(buf)
        return out

    # -- randomized rounding ----------------------------------------------------------------
    def completion_sample(self, Lbuf, k, seed, col0=0):
        """``L^-T g_j`` for the samples j = col0 .. col0+k-1 under ``seed`` (``smcp_csp_sample``), with L from
        ``completion``: an n x k host array, rows in the internal order, columns with covariance the max-det
        completion."""
        n, k, nblk = self.symb.n, int(k), self.symb.nblk
        count = max(1, -(-(n * k) // nblk))
        buf = self.alloc_batch(count)
        try:
            _ck(self.lib, self.lib.smcp_csp_sample(self.sym, Lbuf, int(seed), int(col0), buf, n, k))
            out = self.get_batch(buf, count).reshape(-1)[:n * k].reshape(n, k, order="F")
        finally:
            self.free_batch(buf)
        TRAFFIC["d2h"] += 8 * n * k
        return out

    def round_pm1(self, Lbuf, crow, ccol, cval, trials, seed, chunk=0):
        """``trials`` +-1 roundings sign(L^-T g_t) against the objective given by its lower-triangular entries
        (``crow``, ``ccol`` in internal coordinates, ``cval``) on the device (``smcp_round_pm1``).  Returns
        ``(values, x, best)``: the value of every trial, the int8 sign vector of the best one (internal order)
        and its index."""
        crow, ccol = _i64(crow), _i64(ccol)
        cval = np.ascontiguousarray(cval, dtype=np.float64)
        if not len(crow) == len(ccol) == len(cval):
            raise ValueError("crow, ccol and cval must have the same length")
        values = np.empty(max(0, int(trials)))
        x = np.empty(self.symb.n, dtype=np.int8)
        best = C.c_int64()
        _ck(self.lib, self.lib.smcp_round_pm1(self.sym, Lbuf, int(seed), int(trials), int(chunk), len(cval), crow, ccol,
                                              cval, values, x, C.byref(best)))
        TRAFFIC["h2d"] += 24 * len(cval)
        TRAFFIC["d2h"] += 8 * len(values) + len(x)
        return values, x, best.value

    def round_pm1_ls(self, Lbuf, crow, ccol, cval, trials, seed, chunk=0, max_flips=None, tol=1e-12):
        """``round_pm1`` with the one-flip local search run on every trial on the device (``smcp_round_pm1_ls``;
        ``max_flips`` None: n).  Returns ``(values0, values, flips, x, best)``: the value of every trial before and
        after the search, its number of flips, and the int8 sign vector (internal order) and index of the best
        searched trial."""
        crow, ccol = _i64(crow), _i64(ccol)
        cval = np.ascontiguousarray(cval, dtype=np.float64)
        if not len(crow) == len(ccol) == len(cval):
            raise ValueError("crow, ccol and cval must have the same length")
        n = self.symb.n
        max_flips = n if max_flips is None else int(max_flips)
        nt = max(0, int(trials))
        values0, values, flips = np.empty(nt), np.empty(nt), np.empty(nt, dtype=np.int64)
        x = np.empty(n, dtype=np.int8)
        best = C.c_int64()
        _ck(self.lib, self.lib.smcp_round_pm1_ls(self.sym, Lbuf, int(seed), int(trials), int(chunk), len(cval), crow, ccol, cval,
                                                 max_flips, float(tol), values0, values, x, C.byref(best), flips))
        TRAFFIC["h2d"] += 24 * len(cval)
        TRAFFIC["d2h"] += 24 * nt + n
        return values0, values, flips, x, best.value

    def pm1_local_search(self, x, crow, ccol, cval, max_flips=None, tol=1e-12):
        """One-flip local search of the rows of the k x n +-1 array ``x`` against the objective given by its entries
        (``crow``, ``ccol``, ``cval``, in the coordinates of x) on the device (``smcp_pm1_local_search``;
        ``max_flips`` None: n).  Returns ``(x, values, flips)``: the searched int8 vectors (a new array), their
        values and their numbers of flips."""
        crow, ccol = _i64(crow), _i64(ccol)
        cval = np.ascontiguousarray(cval, dtype=np.float64)
        if not len(crow) == len(ccol) == len(cval):
            raise ValueError("crow, ccol and cval must have the same length")
        x = np.array(x, dtype=np.int8, order="C", ndmin=2)
        k, n = x.shape
        max_flips = n if max_flips is None else int(max_flips)
        values, flips = np.empty(k), np.empty(k, dtype=np.int64)
        _ck(self.lib, self.lib.smcp_pm1_local_search(self.ctx.h, n, k, x, len(cval), crow, ccol, cval, max_flips, float(tol),
                                                     values, flips))
        TRAFFIC["h2d"] += 24 * len(cval) + 8 * x.size
        TRAFFIC["d2h"] += 8 * x.size + 16 * k
        return x, values, flips

    def round_pm1_tabu(self, Lbuf, crow, ccol, cval, trials, seed, tabu_iters, tenure, chunk=0, max_flips=0, tol=1e-12):
        """``round_pm1_ls`` followed by ``tabu_iters`` moves of tabu search (tabu tenure ``tenure``) on every trial on
        the device (``smcp_round_pm1_tabu``; the one-flip search runs only when ``max_flips`` > 0, None: n).  Returns
        ``(values0, values1, values, flips, moves, best_iter, x, best)``: the value of every trial as rounded, before
        and after the tabu search, its numbers of flips and moves and the move count of its returned vector, and the
        int8 sign vector (internal order) and index of the best trial."""
        crow, ccol = _i64(crow), _i64(ccol)
        cval = np.ascontiguousarray(cval, dtype=np.float64)
        if not len(crow) == len(ccol) == len(cval):
            raise ValueError("crow, ccol and cval must have the same length")
        n = self.symb.n
        max_flips = n if max_flips is None else int(max_flips)
        nt = max(0, int(trials))
        values0, values1, values = np.empty(nt), np.empty(nt), np.empty(nt)
        flips, moves, best_iter = (np.empty(nt, dtype=np.int64) for _ in range(3))
        x = np.empty(n, dtype=np.int8)
        best = C.c_int64()
        _ck(self.lib, self.lib.smcp_round_pm1_tabu(self.sym, Lbuf, int(seed), int(trials), int(chunk), len(cval), crow, ccol,
                                                   cval, max_flips, float(tol), values0, values, x, C.byref(best), flips,
                                                   int(tabu_iters), int(tenure), values1, moves, best_iter))
        TRAFFIC["h2d"] += 24 * len(cval)
        TRAFFIC["d2h"] += 48 * nt + n
        return values0, values1, values, flips, moves, best_iter, x, best.value

    def pm1_tabu_search(self, x, crow, ccol, cval, iters, tenure):
        """Tabu search (``iters`` moves, tabu tenure ``tenure``) of the rows of the k x n +-1 array ``x`` against the
        objective given by its entries (in the coordinates of x) on the device (``smcp_pm1_tabu_search``).  Returns
        ``(x, values, moves, best_iter)``: the returned int8 vectors (a new array), their values, the numbers of moves
        made and the move count of each returned vector."""
        crow, ccol = _i64(crow), _i64(ccol)
        cval = np.ascontiguousarray(cval, dtype=np.float64)
        if not len(crow) == len(ccol) == len(cval):
            raise ValueError("crow, ccol and cval must have the same length")
        x = np.array(x, dtype=np.int8, order="C", ndmin=2)
        k, n = x.shape
        values, moves, best_iter = np.empty(k), np.empty(k, dtype=np.int64), np.empty(k, dtype=np.int64)
        _ck(self.lib, self.lib.smcp_pm1_tabu_search(self.ctx.h, n, k, x, len(cval), crow, ccol, cval, int(iters), int(tenure),
                                                    values, moves, best_iter))
        TRAFFIC["h2d"] += 24 * len(cval) + 8 * x.size
        TRAFFIC["d2h"] += 8 * x.size + 24 * k
        return x, values, moves, best_iter

    # -- low-rank solve ----------------------------------------------------------------------
    def lowrank_solve(self, crow, ccol, cval, b, rank, seed, max_sweeps, tol):
        """Mixing-method solve of min C . V V^T s.t. ||v_i||^2 = b_i on the device (``smcp_lowrank_solve``; C given by
        its entries, b per vertex).  Returns ``(V, f, y, sweeps, colors)``: the n x rank factor, the objective after
        0 .. sweeps sweeps, y_i = (C_ii b_i + <v_i, w_i>) / b_i, the number of sweeps and of colours."""
        crow, ccol = _i64(crow), _i64(ccol)
        cval = np.ascontiguousarray(cval, dtype=np.float64)
        b = np.ascontiguousarray(b, dtype=np.float64)
        if not len(crow) == len(ccol) == len(cval):
            raise ValueError("crow, ccol and cval must have the same length")
        n, r, max_sweeps = len(b), int(rank), int(max_sweeps)
        V = np.empty((n, max(r, 0)))
        f = np.empty(max(max_sweeps, 0) + 1)
        y = np.empty(n)
        sweeps, colors = C.c_int64(), C.c_int64()
        _ck(self.lib, self.lib.smcp_lowrank_solve(self.ctx.h, n, r, len(cval), crow, ccol, cval, b, int(seed), max_sweeps,
                                                  float(tol), V, f, y, C.byref(sweeps), C.byref(colors)))
        TRAFFIC["h2d"] += 24 * len(cval) + 8 * n
        TRAFFIC["d2h"] += 8 * V.size + 8 * (sweeps.value + 1) + 8 * n
        return V, f[:sweeps.value + 1].copy(), y, sweeps.value, colors.value

    def round_pm1_factor(self, V, crow, ccol, cval, trials, seed, chunk=0, max_flips=0, tol=1e-12, tabu_iters=0, tenure=0):
        """``trials`` +-1 roundings sign(V g_t) of the n x r factor V against the objective given by its entries (in the
        coordinates of V) on the device (``smcp_round_pm1_factor``), with the one-flip search when ``max_flips`` > 0
        and the tabu search when ``tabu_iters`` > 0.  Returns ``(values0, values1, values, flips, moves, best_iter, x,
        best)`` as ``round_pm1_tabu``; the outputs of a search that does not run are None."""
        crow, ccol = _i64(crow), _i64(ccol)
        cval = np.ascontiguousarray(cval, dtype=np.float64)
        if not len(crow) == len(ccol) == len(cval):
            raise ValueError("crow, ccol and cval must have the same length")
        V = np.ascontiguousarray(V, dtype=np.float64)
        n, r = V.shape
        nt = max(0, int(trials))
        search, tabu = int(max_flips) > 0 or int(tabu_iters) > 0, int(tabu_iters) > 0
        values = np.empty(nt)
        values0, flips = (np.empty(nt), np.empty(nt, dtype=np.int64)) if search else (None, None)
        values1, moves, best_iter = (np.empty(nt), np.empty(nt, dtype=np.int64), np.empty(nt, dtype=np.int64)) if tabu \
            else (None, None, None)
        x = np.empty(n, dtype=np.int8)
        best = C.c_int64()

        def ptr(a):
            return None if a is None else a.ctypes.data

        _ck(self.lib, self.lib.smcp_round_pm1_factor(self.ctx.h, n, r, V, int(seed), int(trials), int(chunk), len(cval), crow,
                                                     ccol, cval, int(max_flips), float(tol), int(tabu_iters), int(tenure),
                                                     ptr(values0), ptr(values1), values, x, C.byref(best), ptr(flips),
                                                     ptr(moves), ptr(best_iter)))
        TRAFFIC["h2d"] += 24 * len(cval) + 8 * V.size
        TRAFFIC["d2h"] += 8 * nt * (1 + 2 * search + 3 * tabu) + n
        return values0, values1, values, flips, moves, best_iter, x, best.value

    def cholesky_batch(self, buf, count):
        info = np.zeros(count, dtype=np.int32)
        _ck(self.lib, self.lib.smcp_csp_cholesky(self.sym, buf, int(count), info))
        return info

    def completion_batch(self, buf, count):
        info = np.zeros(count, dtype=np.int32)
        _ck(self.lib, self.lib.smcp_csp_completion(self.sym, buf, int(count), info))
        return info

    def llt_batch(self, buf, count):
        _ck(self.lib, self.lib.smcp_csp_llt(self.sym, buf, int(count)))

    def projected_inverse_batch(self, buf, count):
        _ck(self.lib, self.lib.smcp_csp_projected_inverse(self.sym, buf, int(count)))

    def hessian_batch(self, tok, buf, count, inv):
        _ck(self.lib, self.lib.smcp_hess_apply(tok, buf, int(count), int(bool(inv))))

    # -- hessian ----------------------------------------------------------------------
    def hessian_factor(self, Lbuf, Ybuf):
        if self._tok is not None:
            self.lib.smcp_hess_destroy(self._tok)
            self._tok = None
        h = C.c_void_p()
        _ck(self.lib, self.lib.smcp_hess_create(self.sym, Lbuf, Ybuf, C.byref(h)))
        self._tok = h
        return h

    def hessian_apply(self, tok, bufs, inv, adj=None):
        for b in bufs:
            if adj is None:
                _ck(self.lib, self.lib.smcp_hess_apply(tok, b, 1, int(bool(inv))))
            else:
                _ck(self.lib, self.lib.smcp_hess_apply_half(tok, b, 1, int(bool(inv)), int(bool(adj))))

    # -- operator ---------------------------------------------------------------------
    def set_operator(self, Av, Ns):
        import scipy.sparse as sp
        Av = sp.csc_matrix(Av)
        Av.sort_indices()
        symb = self.symb
        self.m, self.Ns = Av.shape[1], int(Ns)
        colptr, rowind = _i64(Av.indptr), _i64(Av.indices)
        vals = np.ascontiguousarray(Av.data, dtype=np.float64)
        h = C.c_void_p()
        _ck(self.lib, self.lib.smcp_op_create(self.sym, self.m, self.Ns, colptr, rowind, vals, C.byref(h)))
        self._op = h
        if self.Ns:
            ri = symb.iperm[symb.Ip[rowind]]
            ci = symb.iperm[symb.Jp[rowind]]
            _ck(self.lib, self.lib.smcp_op_set_entry_coords(h, _i64(ri), _i64(ci)))

    def dense_rows(self):
        """Rows of the dense constraint copy on the device: 0 (no dense constraint), ``symb.nblk`` (full
        copy) or the number of rows any constraint touches (support copy)."""
        out = C.c_int64()
        _ck(self.lib, self.lib.smcp_op_dense_rows(self._op, C.byref(out)))
        return out.value

    def Amap(self, buf):
        TRAFFIC["d2h"] += 8 * self.m
        out = np.empty(self.m)
        _ck(self.lib, self.lib.smcp_op_amap(self._op, buf, -1, out))
        return out

    def Amap_col(self, buf, i):
        out = np.empty(1)
        _ck(self.lib, self.lib.smcp_op_amap(self._op, buf, int(i), out))
        return float(out[0])

    def Aadj(self, y):
        TRAFFIC["h2d"] += 8 * self.m
        p = self._alloc(False)
        _ck(self.lib, self.lib.smcp_op_aadj(self._op, np.ascontiguousarray(y, dtype=np.float64), p))
        return p

    # -- Schur complement -------------------------------------------------------------
    def schur_assemble(self, tok, j0=0, j1=None):
        _ck(self.lib, self.lib.smcp_kkt_assemble(self._op, tok, int(j0), int(self.m if j1 is None else j1)))

    def schur_factor(self, tok):
        info = np.zeros(1, dtype=np.int32)
        if self.comm is None or self.comm[1] == 1:
            self.schur_assemble(tok)
            _ck(self.lib, self.lib.smcp_kkt_factor(self._op, info))
        else:
            rank, nranks, block = self.comm
            _ck(self.lib, self.lib.smcp_kkt_assemble_cyclic(self._op, tok, block, rank, nranks))
            if block % 128 == 0:
                # block-cyclic Cholesky: owners factor their column blocks and broadcast the
                # panels (NCCL); no gather of the unfactored H is needed
                _ck(self.lib, self.lib.smcp_kkt_factor_block(self._op, block, rank, nranks, info))
            else:
                _ck(self.lib, self.lib.smcp_kkt_allgather(self._op, block, rank, nranks))
                _ck(self.lib, self.lib.smcp_kkt_factor(self._op, info))
        if info[0]:
            raise ArithmeticError("Schur complement is not positive definite (info=%d)" % info[0])

    # -- kktsolver='qr' in SYRK form (solvers.py:413-475) ---------------------------------------
    def schur_factor_qr(self, tok):
        info = np.zeros(1, dtype=np.int32)
        _ck(self.lib, self.lib.smcp_kkt_assemble_syrk(self._op, tok))
        _ck(self.lib, self.lib.smcp_kkt_factor(self._op, info))
        if info[0]:
            raise ArithmeticError("Z = G(A) is rank deficient (info=%d)" % info[0])

    # -- kktsolver='qr' in Householder form (options['qr_method'] = 'householder') -------------------
    def schur_factor_householder(self, tok):
        """Zw = Q1 R on the device: Q1 replaces Zw, L = R^T (diag >= 0) becomes the factor of H."""
        info = np.zeros(1, dtype=np.int32)
        _ck(self.lib, self.lib.smcp_kkt_factor_qr(self._op, tok, info))
        if info[0]:
            raise ArithmeticError("Z = G(A) is rank deficient (info=%d)" % info[0])

    def qr_solve(self, g_buf, r):
        """y = H^-1 (r + Z^T g) and X = Z y - g through Q1 and L (``smcp_kkt_qr_solve``)."""
        TRAFFIC["h2d"] += 8 * self.m
        TRAFFIC["d2h"] += 8 * self.m
        y = np.empty(self.m)
        p = self._alloc(False)
        try:
            _ck(self.lib, self.lib.smcp_kkt_qr_solve(self._op, g_buf, np.ascontiguousarray(r, dtype=np.float64).ravel(), y, p))
        except DeviceError:
            self.release(p)
            raise
        return y, p

    def gram_factor(self):
        """Cholesky factor of the Gram matrix <A_i, A_j> (trace inner product) of the constraints: the
        normal equations of the least-norm start of ``SDP.solve_phase1`` (``base.py:383-396``)."""
        info = np.zeros(1, dtype=np.int32)
        _ck(self.lib, self.lib.smcp_kkt_assemble_syrk(self._op, None))
        _ck(self.lib, self.lib.smcp_kkt_factor(self._op, info))
        if info[0]:
            raise ArithmeticError("the constraint matrices are linearly dependent (info=%d)" % info[0])

    def z_tmul(self, buf):
        TRAFFIC["d2h"] += 8 * self.m
        out = np.empty(self.m)
        _ck(self.lib, self.lib.smcp_kkt_z_tmul(self._op, buf, out))
        return out

    def z_mul(self, y):
        TRAFFIC["h2d"] += 8 * self.m
        p = self._alloc(False)
        _ck(self.lib, self.lib.smcp_kkt_z_mul(self._op, np.ascontiguousarray(y, dtype=np.float64), p))
        return p

    def schur_solve(self, y):
        TRAFFIC["h2d"] += 8 * self.m
        TRAFFIC["d2h"] += 8 * self.m
        y = np.array(y, dtype=np.float64).ravel()
        _ck(self.lib, self.lib.smcp_kkt_solve(self._op, y))
        return y

    def get_H(self):
        H = np.empty((self.m, self.m), order="F")
        _ck(self.lib, self.lib.smcp_kkt_get_H(self._op, H.reshape(-1, order="F")))
        return H
