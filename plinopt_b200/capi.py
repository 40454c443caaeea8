"""ctypes binding of the C ABI declared in include/plinopt_b200.h.

This is the same binding a reference maintainer would write (INTEGRATION.md):
plain pointers and sizes, caller-owned numpy buffers.  The library is the
product: if libplinopt_b200.so is missing or no CUDA device is visible every
compute call raises -- there is no CPU fallback.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libplinopt_b200.so")

OK = 0
E_ARG, E_CUDA, E_RANGE, E_SHAPE, E_NODEVICE = -1, -2, -3, -4, -5
MEASURE_NNZ, MEASURE_G2 = 0, 3
MODE_EXHAUSTIVE, MODE_PHILOX = 0, 1
NO_INDEX = 2 ** 64 - 1

# every symbol include/plinopt_b200.h declares (checked by tests/test_capi_symbols.py)
SYMBOLS = [
    "plo_release_workspace", "plo_comm_nccl_version", "plo_comm_unique_id", "plo_comm_create", "plo_comm_rank", "plo_comm_size", "plo_comm_allreduce_i64", "plo_comm_destroy", "plo_set_sweep_devices", "plo_set_orbit_any_shape", "plo_orbit_sweep_devices", "plo_lincomb_search_devices", "plo_mmcheck_batch_devices", "plo_factor_sweep_devices",
    "plo_version", "plo_device_count", "plo_set_device", "plo_last_error",
    "plo_lincomb_search", "plo_lincomb_search_batch", "plo_lincomb_quad", "plo_lincomb_plan_create", "plo_lincomb_plan_run", "plo_lincomb_plan_run_range",
    "plo_lincomb_plan_result", "plo_lincomb_plan_candidates", "plo_lincomb_plan_launches", "plo_lincomb_plan_destroy",
    "plo_orbit_sweep", "plo_orbit_decode", "plo_orbit_space", "plo_orbit_table", "plo_orbit_plan_create",
    "plo_orbit_table_modp", "plo_orbit_sweep64", "plo_orbit_table64", "plo_orbit_plan_run", "plo_orbit_plan_result", "plo_orbit_plan_launches", "plo_orbit_plan_pack", "plo_orbit_plan_kernel", "plo_orbit_magnitude_bounds", "plo_orbit_plan_survivors", "plo_selftest_matrix_index", "plo_orbit_plan_destroy",
    "plo_orbit_plan_create_quad", "plo_orbit_table_quad", "plo_growth_factors_quad", "plo_mmchecker_quad", "plo_orbiter_quad", "plo_orbiter_progress_quad",
    "plo_growth_G2", "plo_mmcheck_batch", "plo_mmcheck_plan_create", "plo_mmcheck_plan_run",
    "plo_mmcheck_plan_result", "plo_mmcheck_plan_launches", "plo_mmcheck_plan_encoding", "plo_mmcheck_plan_input_bits", "plo_mmcheck_encode_check", "plo_mmcheck_plan_destroy", "plo_measure_peaks", "plo_measure_issue_peak",
    "plo_sparsifier", "plo_orbiter", "plo_orbiter_progress", "plo_orbiter_modp", "plo_mmchecker", "plo_mmchecker_bits", "plo_LRP2MM", "plo_slp_build", "plo_slp_export", "plo_slp_free",
    "plo_factor_sweep", "plo_factor_decode", "plo_factor_plan_create", "plo_factor_plan_run", "plo_factor_plan_result",
    "plo_factor_plan_launches", "plo_factor_plan_destroy", "plo_factorizer", "plo_dependency_explore", "plo_depender", "plo_negater", "plo_rotater", "plo_growth_factors",
]


class PloError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"plinopt_b200 error {code}: {msg}")
        self.code = code


class OrbitBest(C.Structure):
    _fields_ = [("score", C.c_double), ("nnz", C.c_uint32), ("nno", C.c_uint32), ("index", C.c_uint64)]


class Csr(C.Structure):
    _fields_ = [("rows", C.c_int), ("cols", C.c_int), ("ptr", C.c_void_p), ("col", C.c_void_p), ("val", C.c_void_p)]


_lib = None


def lib():
    """Loads the shared library (raises if it was not built: no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PloError(E_NODEVICE, f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
        L = C.CDLL(LIB_PATH)
        L.plo_last_error.restype = C.c_char_p
        L.plo_orbit_space.restype = C.c_uint64
        L.plo_lincomb_plan_candidates.restype = C.c_uint64
        L.plo_lincomb_plan_candidates.argtypes = [C.c_void_p]
        L.plo_lincomb_plan_launches.argtypes = [C.c_void_p]
        L.plo_lincomb_plan_destroy.argtypes = [C.c_void_p]
        L.plo_lincomb_plan_destroy.restype = None
        L.plo_orbit_plan_destroy.argtypes = [C.c_void_p]
        L.plo_orbit_plan_destroy.restype = None
        L.plo_orbit_plan_launches.argtypes = [C.c_void_p]
        L.plo_mmcheck_plan_destroy.argtypes = [C.c_void_p]
        L.plo_mmcheck_plan_destroy.restype = None
        L.plo_mmcheck_plan_launches.argtypes = [C.c_void_p]
        L.plo_orbit_plan_run.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
        L.plo_orbit_plan_result.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(OrbitBest)]
        L.plo_lincomb_plan_run.argtypes = [C.c_void_p, C.c_void_p]
        L.plo_mmcheck_plan_run.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
        _lib = L
    return _lib


def _check(rc, allow=()):
    if rc != 0 and rc not in allow:
        raise PloError(rc, lib().plo_last_error().decode("utf-8", "replace"))
    return rc


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def device_count():
    return lib().plo_device_count()


def set_device(d):
    _check(lib().plo_set_device(int(d)))


# --------------------------------------------------------------------------
# sparsifier candidate search
# --------------------------------------------------------------------------
def lincomb_search(p, TM, off, coeffs, prev_rows=None, init_rl=-1, init_cl=-1):
    """One (block,num) step: returns (best_rl, best_cl, best_index or None)."""
    TM = _i64(TM); coeffs = _i64(coeffs)
    n, m = TM.shape
    prev = _i64(prev_rows) if prev_rows is not None and len(prev_rows) else None
    nprev = 0 if prev is None else prev.shape[0]
    rl, cl, idx = C.c_int(), C.c_int(), C.c_uint64()
    f = lib().plo_lincomb_search
    f.argtypes = [C.c_uint32, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                  C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_uint64)]
    _check(f(int(p), n, m, _ptr(TM), int(off), len(coeffs), _ptr(coeffs), nprev, _ptr(prev), int(init_rl), int(init_cl),
             C.byref(rl), C.byref(cl), C.byref(idx)))
    return rl.value, cl.value, (None if idx.value == NO_INDEX else idx.value)


REDUCE_MIN, REDUCE_MAX = 0, 1


class Comm:
    """The engine's own NCCL communicator (plo_comm_*): one rank per GPU and process.  `exchange(id_or_None)` is whatever hands rank 0's
    128-byte unique id to the other ranks (bench.py: a torch.distributed broadcast) -- the engine does the collective itself."""

    def __init__(self, rank, world, exchange):
        ident = np.zeros(128, dtype=np.uint8)
        if rank == 0:
            _check(lib().plo_comm_unique_id(_ptr(ident)))
        ident = np.frombuffer(bytes(exchange(ident.tobytes() if rank == 0 else None)), dtype=np.uint8).copy()
        self._h = C.c_void_p()
        f = lib().plo_comm_create
        f.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_void_p]
        _check(f(C.byref(self._h), rank, world, _ptr(ident)))
        self.rank, self.world = rank, world

    def allreduce_i64(self, device_ptr, count, op=REDUCE_MIN, stream=0):
        f = lib().plo_comm_allreduce_i64
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p]
        _check(f(self._h, C.c_void_p(device_ptr), count, op, C.c_void_p(stream)))

    def close(self):
        if self._h:
            f = lib().plo_comm_destroy
            f.argtypes = [C.c_void_p]
            f(self._h)
            self._h = C.c_void_p()


def lincomb_search_devices(ndev, p, TM, off, coeffs, prev_rows=None, init_rl=-1, init_cl=-1):
    """plo_lincomb_search_devices on one problem: (best_rl, best_cl, best_index or None)."""
    TM = _i64(TM); coeffs = _i64(coeffs)
    n, m = TM.shape
    prev = _i64(prev_rows) if prev_rows is not None and len(prev_rows) else None
    nprev = 0 if prev is None else prev.shape[0]
    rl, cl, idx = C.c_int(), C.c_int(), C.c_uint64()
    irl, icl = C.c_int(int(init_rl)), C.c_int(int(init_cl))
    f = lib().plo_lincomb_search_devices
    f.argtypes = [C.c_int, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int),
                  C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_uint64)]
    _check(f(int(ndev), int(p), 1, n, m, _ptr(TM), int(off), len(coeffs), _ptr(coeffs), nprev, _ptr(prev), C.byref(irl), C.byref(icl),
             C.byref(rl), C.byref(cl), C.byref(idx)))
    return rl.value, cl.value, (None if idx.value == NO_INDEX else idx.value)


class QuadProblem(C.Structure):
    _fields_ = [("n", C.c_int), ("off", C.c_int), ("c", C.c_int), ("nprev", C.c_int), ("TM", C.c_void_p), ("coeffs", C.c_void_p),
                ("prev_rows", C.c_void_p), ("seed_vec", C.c_void_p), ("init_rl", C.c_int), ("init_cl", C.c_int), ("nrows", C.c_int),
                ("status", C.c_int), ("rl", C.c_int * 4), ("cl", C.c_int * 4), ("index", C.c_uint64 * 4)]


QUAD_DONE, QUAD_MISS, QUAD_SEED, QUAD_RANGE = 0, 1, 2, 3


def lincomb_quad(p, problems):
    """All rows of one inner block for a list of independent problems (plo_lincomb_quad).  Each problem is a dict with TM (n x m),
    off, coeffs and optionally prev_rows, init_rl, init_cl, seed_vec.  Returns per problem (status, [(rl, cl, index or None), ...])."""
    arr = (QuadProblem * len(problems))()
    keep = []
    m = None
    for q, pr in zip(arr, problems):
        TM = _i64(pr["TM"]); cf = _i64(pr["coeffs"])
        prev = pr.get("prev_rows")
        prev = _i64(prev) if prev is not None and len(prev) else None
        sv = pr.get("seed_vec")
        sv = _i64(sv) if sv is not None else None
        keep += [TM, cf, prev, sv]
        if m is None:
            m = TM.shape[1]
        assert TM.shape[1] == m
        q.n, q.off, q.c, q.nprev = TM.shape[0], int(pr.get("off", 0)), len(cf), (0 if prev is None else prev.shape[0])
        q.TM, q.coeffs, q.prev_rows, q.seed_vec = _ptr(TM), _ptr(cf), _ptr(prev), _ptr(sv)
        q.init_rl, q.init_cl = int(pr.get("init_rl", -1)), int(pr.get("init_cl", -1))
    f = lib().plo_lincomb_quad
    f.argtypes = [C.c_uint32, C.c_int, C.c_int, C.c_void_p]
    _check(f(int(p), int(m), len(problems), C.cast(arr, C.c_void_p)))
    out = []
    for q in arr:
        out.append((q.status, [(q.rl[t], q.cl[t], (None if q.index[t] == NO_INDEX else q.index[t])) for t in range(q.nrows)]))
    return out


class LincombPlan:
    """Device-resident batch of independent searches (plo_lincomb_plan_*)."""

    def __init__(self, p, TM, off, coeffs, prev_rows=None, init_rl=None, init_cl=None):
        TM = _i64(TM); coeffs = _i64(coeffs)
        if TM.ndim == 2:
            TM = TM[None]; coeffs = coeffs[None]
            prev_rows = None if prev_rows is None else _i64(prev_rows)[None]
        self.nbatch, n, m = TM.shape
        prev = _i64(prev_rows) if prev_rows is not None and np.size(prev_rows) else None
        nprev = 0 if prev is None else prev.shape[1]
        irl = None if init_rl is None else _i32(np.broadcast_to(init_rl, (self.nbatch,)))
        icl = None if init_cl is None else _i32(np.broadcast_to(init_cl, (self.nbatch,)))
        self._h = C.c_void_p()
        f = lib().plo_lincomb_plan_create
        f.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                      C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        _check(f(C.byref(self._h), int(p), self.nbatch, n, m, _ptr(TM), int(off), coeffs.shape[1], _ptr(coeffs), nprev,
                 _ptr(prev), _ptr(irl), _ptr(icl)))
        self.candidates = lib().plo_lincomb_plan_candidates(self._h)
        self.launches = lib().plo_lincomb_plan_launches(self._h)

    def run(self, stream=0):
        _check(lib().plo_lincomb_plan_run(self._h, C.c_void_p(stream)))

    def run_range(self, prefix_lo, prefix_hi, stream=0):
        """Only the candidates whose prefix (i*c+j)*c+k is in [prefix_lo, prefix_hi): one shard of the search."""
        f = lib().plo_lincomb_plan_run_range
        f.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
        _check(f(self._h, prefix_lo, prefix_hi, C.c_void_p(stream)))

    def result(self, stream=0):
        rl = np.zeros(self.nbatch, dtype=np.int32); cl = np.zeros(self.nbatch, dtype=np.int32)
        idx = np.zeros(self.nbatch, dtype=np.uint64)
        f = lib().plo_lincomb_plan_result
        f.argtypes = [C.c_void_p] * 5
        _check(f(self._h, C.c_void_p(stream), _ptr(rl), _ptr(cl), _ptr(idx)))
        return rl, cl, idx

    def close(self):
        if self._h:
            lib().plo_lincomb_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# --------------------------------------------------------------------------
# orbit sweep
# --------------------------------------------------------------------------
def set_orbit_any_shape(on):
    """1: orbit shapes without a compiled kernel run on the runtime-shape kernels (process-wide); 0 (default): E_SHAPE."""
    _check(lib().plo_set_orbit_any_shape(int(on)))


def orbit_decode(m, k, n, mode, seed, index):
    U = np.zeros((m, m), dtype=np.int32); V = np.zeros((k, k), dtype=np.int32); W = np.zeros((n, n), dtype=np.int32)
    f = lib().plo_orbit_decode
    f.argtypes = [C.c_int] * 4 + [C.c_uint64, C.c_uint64] + [C.c_void_p] * 3
    _check(f(m, k, n, mode, seed, index, _ptr(U), _ptr(V), _ptr(W)))
    return U, V, W


def orbit_space(m, k, n):
    f = lib().plo_orbit_space
    f.argtypes = [C.c_int] * 3
    return f(m, k, n)


def _best_tuple(b):
    return dict(score=b.score, nnz=b.nnz, nno=b.nno, index=(None if b.index == NO_INDEX else b.index))


def orbit_sweep(mkn, L, R, P, dens, measure, mode, seed, lo, hi, p=0):
    """Host-buffer entry point (copies inside): returns dict(score, nnz, nno, index)."""
    m, k, n = mkn
    L = _i32(L); R = _i32(R); P = _i32(P)
    best = OrbitBest()
    f = lib().plo_orbit_sweep
    f.argtypes = [C.c_uint32] + [C.c_int] * 4 + [C.c_void_p] * 3 + [C.c_int32] * 3 + [C.c_int, C.c_int, C.c_uint64, C.c_uint64,
                  C.c_uint64, C.POINTER(OrbitBest)]
    _check(f(p, m, k, n, L.shape[0], _ptr(L), _ptr(R), _ptr(P), dens[0], dens[1], dens[2], measure, mode, seed, lo, hi, C.byref(best)))
    return _best_tuple(best)


def orbit_sweep_devices(ndev, mkn, L, R, P, dens, measure, mode, seed, lo, hi):
    """One process, `ndev` devices: the sharded form of orbit_sweep (same winner)."""
    m, k, n = mkn
    L = _i32(L); R = _i32(R); P = _i32(P)
    best = OrbitBest()
    f = lib().plo_orbit_sweep_devices
    f.argtypes = [C.c_int] * 5 + [C.c_void_p] * 3 + [C.c_int32] * 3 + [C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(OrbitBest)]
    _check(f(ndev, m, k, n, L.shape[0], _ptr(L), _ptr(R), _ptr(P), dens[0], dens[1], dens[2], measure, mode, seed, lo, hi, C.byref(best)))
    return _best_tuple(best)


def orbit_table(mkn, L, R, P, dens, mode, seed, lo, hi):
    m, k, n = mkn
    L = _i32(L); R = _i32(R); P = _i32(P)
    cnt = hi - lo
    nnz = np.zeros(cnt, dtype=np.uint32); nno = np.zeros(cnt, dtype=np.uint32); g2 = np.zeros(cnt, dtype=np.float64)
    f = lib().plo_orbit_table
    f.argtypes = [C.c_int] * 4 + [C.c_void_p] * 3 + [C.c_int32] * 3 + [C.c_int, C.c_uint64, C.c_uint64, C.c_uint64] + [C.c_void_p] * 3
    _check(f(m, k, n, L.shape[0], _ptr(L), _ptr(R), _ptr(P), dens[0], dens[1], dens[2], mode, seed, lo, hi, _ptr(nnz), _ptr(nno), _ptr(g2)))
    return nnz, nno, g2


def orbit_sweep64(mkn, L, R, P, dens, measure, mode, seed, lo, hi):
    """int64 entries / denominators (plo_orbit_sweep64)."""
    m, k, n = mkn
    L = _i64(L); R = _i64(R); P = _i64(P)
    best = OrbitBest()
    f = lib().plo_orbit_sweep64
    f.argtypes = [C.c_int] * 4 + [C.c_void_p] * 3 + [C.c_int64] * 3 + [C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(OrbitBest)]
    _check(f(m, k, n, L.shape[0], _ptr(L), _ptr(R), _ptr(P), dens[0], dens[1], dens[2], measure, mode, seed, lo, hi, C.byref(best)))
    return _best_tuple(best)


def orbit_table64(mkn, L, R, P, dens, mode, seed, lo, hi):
    m, k, n = mkn
    L = _i64(L); R = _i64(R); P = _i64(P)
    cnt = hi - lo
    nnz = np.zeros(cnt, dtype=np.uint32); nno = np.zeros(cnt, dtype=np.uint32); g2 = np.zeros(cnt, dtype=np.float64)
    f = lib().plo_orbit_table64
    f.argtypes = [C.c_int] * 4 + [C.c_void_p] * 3 + [C.c_int64] * 3 + [C.c_int, C.c_uint64, C.c_uint64, C.c_uint64] + [C.c_void_p] * 3
    _check(f(m, k, n, L.shape[0], _ptr(L), _ptr(R), _ptr(P), dens[0], dens[1], dens[2], mode, seed, lo, hi, _ptr(nnz), _ptr(nno), _ptr(g2)))
    return nnz, nno, g2


def orbit_table_modp(p, mkn, L, R, P, mode, seed, lo, hi):
    """Per-candidate (nnz, nno) over Z/pZ; L, R, P hold residues."""
    m, k, n = mkn
    L = _i32(L); R = _i32(R); P = _i32(P)
    cnt = hi - lo
    nnz = np.zeros(cnt, dtype=np.uint32); nno = np.zeros(cnt, dtype=np.uint32)
    f = lib().plo_orbit_table_modp
    f.argtypes = [C.c_uint32] + [C.c_int] * 4 + [C.c_void_p] * 3 + [C.c_int, C.c_uint64, C.c_uint64, C.c_uint64] + [C.c_void_p] * 2
    _check(f(p, m, k, n, L.shape[0], _ptr(L), _ptr(R), _ptr(P), mode, seed, lo, hi, _ptr(nnz), _ptr(nno)))
    return nnz, nno


def orbit_table_quad(d, mkn, La, Lb, Ra, Rb, Pa, Pb, dens, mode, seed, lo, hi):
    """Per-candidate (nnz, nno, g2) over Q(sqrt d): entry = (a + b.sqrt(d)) / den, a from the `*a` arrays, b from the `*b` arrays
    (int64, layout of orbit_table).  g2 is None for d < 0 (no real embedding)."""
    m, k, n = mkn
    parts = [_i64(x) for x in (La, Lb, Ra, Rb, Pa, Pb)]
    cnt = hi - lo
    nnz = np.zeros(cnt, dtype=np.uint32); nno = np.zeros(cnt, dtype=np.uint32)
    g2 = np.zeros(cnt, dtype=np.float64) if d > 0 else None
    f = lib().plo_orbit_table_quad
    f.argtypes = [C.c_int64] + [C.c_int] * 4 + [C.c_void_p] * 6 + [C.c_int64] * 3 + [C.c_int, C.c_uint64, C.c_uint64, C.c_uint64] + [C.c_void_p] * 3
    _check(f(d, m, k, n, parts[0].shape[0], *(_ptr(x) for x in parts), dens[0], dens[1], dens[2], mode, seed, lo, hi, _ptr(nnz), _ptr(nno), _ptr(g2)))
    return nnz, nno, g2


class OrbitPlan:
    def __init__(self, mkn, L, R, P, dens, measure, mode, seed):
        m, k, n = mkn
        L = _i32(L); R = _i32(R); P = _i32(P)
        self._h = C.c_void_p()
        f = lib().plo_orbit_plan_create
        f.argtypes = [C.POINTER(C.c_void_p)] + [C.c_int] * 4 + [C.c_void_p] * 3 + [C.c_int32] * 3 + [C.c_int, C.c_int, C.c_uint64]
        _check(f(C.byref(self._h), m, k, n, L.shape[0], _ptr(L), _ptr(R), _ptr(P), dens[0], dens[1], dens[2], measure, mode, seed))
        self._describe()

    @classmethod
    def quad(cls, d, mkn, La, Lb, Ra, Rb, Pa, Pb, dens, measure, mode, seed):
        """A plan over Q(sqrt d) (plo_orbit_plan_create_quad); run, result, pack, survivors as for any plan."""
        self = cls.__new__(cls)
        m, k, n = mkn
        parts = [_i64(x) for x in (La, Lb, Ra, Rb, Pa, Pb)]
        self._h = C.c_void_p()
        f = lib().plo_orbit_plan_create_quad
        f.argtypes = [C.POINTER(C.c_void_p), C.c_int64] + [C.c_int] * 4 + [C.c_void_p] * 6 + [C.c_int64] * 3 + [C.c_int, C.c_int, C.c_uint64]
        _check(f(C.byref(self._h), d, m, k, n, parts[0].shape[0], *(_ptr(x) for x in parts), dens[0], dens[1], dens[2], measure, mode, seed))
        self._describe()
        return self

    def _describe(self):
        self.launches = lib().plo_orbit_plan_launches(self._h)
        name = C.create_string_buffer(64)
        lanes = C.c_int(0)
        _check(lib().plo_orbit_plan_kernel(self._h, name, 64, C.byref(lanes)))
        self.kernel, self.lanes = name.value.decode(), lanes.value

    def run(self, lo, hi, stream=0):
        _check(lib().plo_orbit_plan_run(self._h, lo, hi, C.c_void_p(stream)))

    def result(self, stream=0):
        best = OrbitBest()
        _check(lib().plo_orbit_plan_result(self._h, C.c_void_p(stream), C.byref(best)))
        return _best_tuple(best)

    def pack(self, slots_ptr, rank, world, stream=0):
        """Winner of the last run -> slot `rank` of a device table of world x 4 int64 words (see plo_orbit_plan_pack)."""
        f = lib().plo_orbit_plan_pack
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        _check(f(self._h, C.c_void_p(slots_ptr), rank, world, C.c_void_p(stream)))

    def survivors(self, lo, hi, nnz=0, nno=0, score=0.0, capacity=1 << 16):
        """Candidates of [lo,hi) not worse than the threshold (sparsity plans: (nnz, nno); growth-factor plans: score), sorted by
        index: list of dicts with index, nnz, nno, score (= growth factor).  Grows the buffer once if `capacity` was too small."""
        f = lib().plo_orbit_plan_survivors
        f.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(OrbitBest), C.c_uint64, C.POINTER(OrbitBest), C.POINTER(C.c_uint64)]
        thr = OrbitBest(score=score, nnz=nnz, nno=nno, index=0)
        cnt = C.c_uint64(0)
        for _ in range(2):
            buf = (OrbitBest * max(1, capacity))()
            rc = f(self._h, lo, hi, C.byref(thr), capacity, buf, C.byref(cnt))
            if rc == E_RANGE and cnt.value > capacity:
                capacity = cnt.value
                continue
            _check(rc)
            return [_best_tuple(buf[i]) for i in range(cnt.value)]
        _check(rc)

    def survivors_array(self, lo, hi, nnz=0, nno=0, score=0.0, capacity=1 << 16):
        """The same as `survivors` without the per-record Python objects: (count, structured numpy array score/nnz/nno/index).
        Raises PloError(E_RANGE) when `capacity` is too small (the message carries the count)."""
        f = lib().plo_orbit_plan_survivors
        f.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(OrbitBest), C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)]
        thr = OrbitBest(score=score, nnz=nnz, nno=nno, index=0)
        buf = np.zeros(max(1, capacity), dtype=np.dtype([("score", "<f8"), ("nnz", "<u4"), ("nno", "<u4"), ("index", "<u8")]))
        cnt = C.c_uint64(0)
        _check(f(self._h, lo, hi, C.byref(thr), capacity, _ptr(buf), C.byref(cnt)))
        return cnt.value, buf[:cnt.value]

    def close(self):
        if self._h:
            lib().plo_orbit_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def orbit_magnitude_bounds(mkn, L, R, P):
    """(lanes, (bL, bR, bP)): host-only worst-case magnitudes of the transformed entries over the whole orbit."""
    m, k, n = mkn
    L = _i32(L); R = _i32(R); P = _i32(P)
    b = np.zeros(3, dtype=np.int64)
    f = lib().plo_orbit_magnitude_bounds
    f.argtypes = [C.c_int] * 4 + [C.c_void_p] * 4
    rc = f(m, k, n, L.shape[0], _ptr(L), _ptr(R), _ptr(P), _ptr(b))
    if rc < 0:
        _check(rc)
    return rc, tuple(int(x) for x in b)


def growth_G2(L, R, P):
    """G2 of dense double triples; L (batch, r, a), R (batch, r, b), P (batch, c, r)."""
    L = np.ascontiguousarray(L, dtype=np.float64); R = np.ascontiguousarray(R, dtype=np.float64); P = np.ascontiguousarray(P, dtype=np.float64)
    if L.ndim == 2:
        L, R, P = L[None], R[None], P[None]
    batch, r, a = L.shape
    out = np.zeros(batch, dtype=np.float64)
    f = lib().plo_growth_G2
    f.argtypes = [C.c_int] * 5 + [C.c_void_p] * 4
    _check(f(batch, r, a, R.shape[2], P.shape[1], _ptr(L), _ptr(R), _ptr(P), _ptr(out)))
    return out


# --------------------------------------------------------------------------
# MMchecker
# --------------------------------------------------------------------------
class _CsrHolder:
    def __init__(self, rows, cols, ptr, col, val):
        self.ptr = _i64(ptr); self.col = _i32(col); self.val = np.ascontiguousarray(val, dtype=np.uint32)
        self.c = Csr(rows, cols, self.ptr.ctypes.data, self.col.ctypes.data, self.val.ctypes.data)


def mmcheck_batch(p, mkn, r, L, R, P, seed=0, batch=1, ua=None, ub=None):
    """L,R,P = (rows, cols, ptr, col, val) CSR tuples.  Returns (verdict, ok[batch])."""
    m, k, n = mkn
    hl, hr, hp = _CsrHolder(*L), _CsrHolder(*R), _CsrHolder(*P)
    ok = np.zeros(batch, dtype=np.uint8)
    a = None if ua is None else np.ascontiguousarray(ua, dtype=np.uint32)
    b = None if ub is None else np.ascontiguousarray(ub, dtype=np.uint32)
    f = lib().plo_mmcheck_batch
    f.argtypes = [C.c_uint32] + [C.c_int] * 4 + [C.POINTER(Csr)] * 3 + [C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    rc = _check(f(p, m, k, n, r, C.byref(hl.c), C.byref(hr.c), C.byref(hp.c), seed, batch, _ptr(a), _ptr(b), _ptr(ok)), allow=(1, 2, 3))
    return rc, ok


def mmcheck_batch_devices(ndev, p, mkn, r, L, R, P, seed=0, batch=1):
    """plo_mmcheck_batch_devices: the batch split over the first ndev devices.  Returns (verdict, ok[batch])."""
    m, k, n = mkn
    hl, hr, hp = _CsrHolder(*L), _CsrHolder(*R), _CsrHolder(*P)
    ok = np.zeros(batch, dtype=np.uint8)
    f = lib().plo_mmcheck_batch_devices
    f.argtypes = [C.c_int, C.c_uint32] + [C.c_int] * 4 + [C.POINTER(Csr)] * 3 + [C.c_uint64, C.c_int, C.c_void_p]
    rc = _check(f(int(ndev), p, m, k, n, r, C.byref(hl.c), C.byref(hr.c), C.byref(hp.c), seed, batch, _ptr(ok)), allow=(1, 2, 3))
    return rc, ok


def mmcheck_encode_check(p, A, x, groups=1, row_blocks=True):
    """plo_mmcheck_encode_check (host only): y = A.x mod p replayed from the encoded blobs; returns (y, stats dict)."""
    h = _CsrHolder(*A)
    xs = np.ascontiguousarray(x, dtype=np.uint32)
    assert xs.size == A[1]
    y = np.zeros(A[0], dtype=np.uint32)
    st = (C.c_longlong * 9)()
    f = lib().plo_mmcheck_encode_check
    f.argtypes = [C.c_uint32, C.POINTER(Csr), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    _check(f(p, C.byref(h.c), int(groups), int(bool(row_blocks)), _ptr(xs), _ptr(y), C.cast(st, C.c_void_p)))
    keys = ("row_stride", "col_stride", "chunks", "blob_bytes", "plain_entries", "units", "groups", "loads", "tasks")
    return y, dict(zip(keys, [int(v) for v in st]))


class MMcheckPlan:
    def __init__(self, p, mkn, r, L, R, P, batch):
        m, k, n = mkn
        self._keep = (_CsrHolder(*L), _CsrHolder(*R), _CsrHolder(*P))
        self.batch = batch
        self._h = C.c_void_p()
        f = lib().plo_mmcheck_plan_create
        f.argtypes = [C.POINTER(C.c_void_p), C.c_uint32] + [C.c_int] * 4 + [C.POINTER(Csr)] * 3 + [C.c_int]
        _check(f(C.byref(self._h), p, m, k, n, r, C.byref(self._keep[0].c), C.byref(self._keep[1].c), C.byref(self._keep[2].c), batch))
        self.launches = lib().plo_mmcheck_plan_launches(self._h)
        loads, blob, strides = (C.c_int64 * 3)(), (C.c_int64 * 3)(), (C.c_int * 6)()
        g = lib().plo_mmcheck_plan_encoding
        g.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        _check(g(self._h, C.cast(loads, C.c_void_p), C.cast(blob, C.c_void_p), C.cast(strides, C.c_void_p)))
        self.encoding = {"loads": [int(v) for v in loads], "blob_bytes": [int(v) for v in blob],
                         "col_stride": [int(strides[2 * z]) for z in range(3)], "row_stride": [int(strides[2 * z + 1]) for z in range(3)]}

    def run(self, seed, first_sample=0, stream=0):
        _check(lib().plo_mmcheck_plan_run(self._h, seed, first_sample, C.c_void_p(stream)))

    def result(self, stream=0):
        ok = np.zeros(self.batch, dtype=np.uint8)
        v = C.c_int()
        f = lib().plo_mmcheck_plan_result
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]
        _check(f(self._h, C.c_void_p(stream), _ptr(ok), C.byref(v)))
        return v.value, ok

    def close(self):
        if self._h:
            lib().plo_mmcheck_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def measure_peaks(reps=10):
    a, b, c = C.c_double(), C.c_double(), C.c_double()
    f = lib().plo_measure_peaks
    f.argtypes = [C.c_int] + [C.POINTER(C.c_double)] * 3
    _check(f(reps, C.byref(a), C.byref(b), C.byref(c)))
    d = C.c_double()
    g = lib().plo_measure_issue_peak
    g.argtypes = [C.c_int, C.POINTER(C.c_double)]
    _check(g(reps, C.byref(d)))
    return dict(imad_per_s=a.value, dfma_per_s=b.value, ialu_pairs_per_s=c.value, issue_inst_per_s=d.value)


# --------------------------------------------------------------------------
# host-level entry points (reference drivers restated around the kernels)
# --------------------------------------------------------------------------
class OrbiterReport(C.Structure):
    _fields_ = [("init_nnz", C.c_uint32), ("init_nno", C.c_uint32), ("init_score", C.c_double), ("best", OrbitBest),
                ("improved", C.c_int), ("mm_verdict", C.c_int), ("m", C.c_int), ("k", C.c_int), ("n", C.c_int)]


def _numden(M):
    """list of rows of Fraction / int -> (num, den) int64 arrays."""
    from fractions import Fraction
    r, c = len(M), len(M[0])
    num = np.zeros((r, c), dtype=np.int64); den = np.ones((r, c), dtype=np.int64)
    for i in range(r):
        for j in range(c):
            v = Fraction(M[i][j])
            num[i, j] = v.numerator; den[i, j] = v.denominator
    return num, den


def _fractions(num, den):
    from fractions import Fraction
    return [[Fraction(int(num[i, j]), int(den[i, j])) for j in range(num.shape[1])] for i in range(num.shape[0])]


def sparsifier(M, q=0, blocksize=4, maxnumcoeff=11, initial_elimination=True, log_fd=-1):
    """blockSparsifier through the GPU search.  Returns (CoB, Res, consistent, stats dict)."""
    num, den = _numden(M)
    r, c = num.shape
    cn = np.zeros((c, c), dtype=np.int64); cd = np.ones((c, c), dtype=np.int64)
    rn = np.zeros((r, c), dtype=np.int64); rd = np.ones((r, c), dtype=np.int64)
    ok = C.c_int(0)
    stats = np.zeros(3, dtype=np.uint64)
    f = lib().plo_sparsifier
    f.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 4 + [C.POINTER(C.c_int), C.c_void_p, C.c_int]
    _check(f(q, r, c, _ptr(num), _ptr(den), blocksize, maxnumcoeff, 1 if initial_elimination else 0, _ptr(cn), _ptr(cd), _ptr(rn), _ptr(rd),
             C.byref(ok), _ptr(stats), log_fd))
    st = dict(candidates=int(stats[0]), searches=int(stats[1]), fallbacks=int(stats[2]))
    if q == 0:
        return _fractions(cn, cd), _fractions(rn, rd), bool(ok.value), st
    return cn.tolist(), rn.tolist(), bool(ok.value), st


def _triple(d, L, R, P):
    """The arguments an entry point and its _quad twin share.  d None: L, R, P are lists of rows of Fraction, passed as (num, den)
    per matrix.  Otherwise each is a pair (rational part, sqrt(d) part), passed as (an, ad, bn, bd) per matrix after the leading
    int64 d.  Returns (leading arguments, their ctypes, the arrays, the rational parts)."""
    if d is None:
        return [], [], [a for M in (L, R, P) for a in _numden(M)], (L, R, P)
    return [d], [C.c_int64], [a for M in (L, R, P) for part in M for a in _numden(part)], tuple(M[0] for M in (L, R, P))


def _report(rep):
    return dict(init_nnz=rep.init_nnz, init_nno=rep.init_nno, init_score=rep.init_score, best=_best_tuple(rep.best),
                improved=bool(rep.improved), mm_verdict=rep.mm_verdict, mkn=(rep.m, rep.k, rep.n))


def _orbiter(d, L, R, P, measure, mode, seed, loops):
    lead, types, arrs, (La, Ra, Pa) = _triple(d, L, R, P)
    outs = [np.zeros_like(a) for a in arrs]
    rep = OrbiterReport()
    f = lib().plo_orbiter if d is None else lib().plo_orbiter_quad
    f.argtypes = types + [C.c_int, C.c_int, C.c_uint64, C.c_uint64] + [C.c_int] * 4 + [C.c_void_p] * (2 * len(arrs)) + [C.POINTER(OrbiterReport)]
    _check(f(*lead, measure, mode, seed, loops, len(La), len(La[0]), len(Ra[0]), len(Pa), *(_ptr(x) for x in arrs + outs), C.byref(rep)))
    mats = [_fractions(outs[t], outs[t + 1]) for t in range(0, len(outs), 2)]
    return (*(mats if d is None else zip(mats[::2], mats[1::2])), _report(rep))


def _orbiter_progress(d, L, R, P, measure, mode, seed, loops, capacity):
    lead, types, arrs, (La, Ra, Pa) = _triple(d, L, R, P)
    buf = (OrbitBest * capacity)()
    cnt = C.c_uint64(0)
    f = lib().plo_orbiter_progress if d is None else lib().plo_orbiter_progress_quad
    f.argtypes = types + [C.c_int, C.c_int, C.c_uint64, C.c_uint64] + [C.c_int] * 4 + [C.c_void_p] * len(arrs) + [C.c_uint64, C.POINTER(OrbitBest), C.POINTER(C.c_uint64)]
    _check(f(*lead, measure, mode, seed, loops, len(La), len(La[0]), len(Ra[0]), len(Pa), *(_ptr(x) for x in arrs), capacity, buf, C.byref(cnt)))
    return [_best_tuple(buf[i]) for i in range(cnt.value)]


def orbiter(L, R, P, measure=MEASURE_NNZ, mode=MODE_PHILOX, seed=0, loops=100):
    """Orbiter over Q.  Returns (Lj, Rg, hP, report dict)."""
    return _orbiter(None, L, R, P, measure, mode, seed, loops)


def orbiter_progress(L, R, P, measure=MEASURE_NNZ, mode=MODE_PHILOX, seed=0, loops=100, capacity=256):
    """The deterministic '# Found opt:' records (plo_orbiter_progress): list of dicts in increasing index order."""
    return _orbiter_progress(None, L, R, P, measure, mode, seed, loops, capacity)


def orbiter_modp(L, R, P, q, mode=MODE_PHILOX, seed=0, loops=100):
    """plo_orbiter_modp: returns (Lj, Rg, hP) as residue lists and the report dict."""
    Ln, Ld = _numden(L); Rn, Rd = _numden(R); Pn, Pd = _numden(P)
    oL, oR, oP = np.zeros_like(Ln), np.zeros_like(Rn), np.zeros_like(Pn)
    rep = OrbiterReport()
    f = lib().plo_orbiter_modp
    f.argtypes = [C.c_uint64, C.c_int, C.c_uint64, C.c_uint64] + [C.c_int] * 4 + [C.c_void_p] * 9 + [C.POINTER(OrbiterReport)]
    _check(f(q, mode, seed, loops, Ln.shape[0], Ln.shape[1], Rn.shape[1], Pn.shape[0], _ptr(Ln), _ptr(Ld), _ptr(Rn), _ptr(Rd), _ptr(Pn), _ptr(Pd),
             _ptr(oL), _ptr(oR), _ptr(oP), C.byref(rep)))
    report = dict(init=(rep.init_nnz, rep.init_nno), best=_best_tuple(rep.best), improved=bool(rep.improved), mm_verdict=rep.mm_verdict,
                  mkn=(rep.m, rep.k, rep.n))
    return oL.tolist(), oR.tolist(), oP.tolist(), report


def _mmchecker(name, lead, types, arrs, parts, with_nprimes=True):
    """plo_mmchecker, plo_mmchecker_bits or plo_mmchecker_quad: (verdict, (nnz, nno), number of primes used)."""
    cnt = np.zeros(2, dtype=np.uint32)
    npr = C.c_int()
    f = getattr(lib(), name)
    f.argtypes = types + [C.c_int] * 6 + [C.c_void_p] * (len(arrs) + 1) + [C.POINTER(C.c_int)] * with_nprimes
    dims = [x for M in parts for x in (len(M), len(M[0]))]
    rc = _check(f(*lead, *dims, *(_ptr(x) for x in arrs), _ptr(cnt), *[C.byref(npr)] * with_nprimes), allow=(1, 2, 3))
    return rc, (int(cnt[0]), int(cnt[1])), npr.value


def mmchecker(L, R, P, modulus=0, seed=0, batch=32):
    """fMMchecker on dense rational matrices.  Returns (verdict, (nnz, nno))."""
    _, _, arrs, parts = _triple(None, L, R, P)
    return _mmchecker("plo_mmchecker", [modulus, seed, batch], [C.c_uint64, C.c_uint64, C.c_int], arrs, parts, with_nprimes=False)[:2]


def mmchecker_bits(L, R, P, modulus=0, bitsize=32, seed=0, batch=32):
    """plo_mmchecker_bits: over Q (modulus 0) the decision is exact at every sampled point with `bitsize`-bit integer coordinates.
    Returns (verdict, (nnz, nno), number of primes used)."""
    _, _, arrs, parts = _triple(None, L, R, P)
    return _mmchecker("plo_mmchecker_bits", [modulus, bitsize, seed, batch], [C.c_uint64, C.c_int, C.c_uint64, C.c_int], arrs, parts)


def mmchecker_quad(d, L, R, P, bitsize=32, seed=0, batch=32):
    """plo_mmchecker_quad: the exact check over Q(sqrt d); L, R, P are pairs (rational part, sqrt(d) part) of lists of rows of
    Fraction.  Returns (verdict, (nnz, nno), number of primes used)."""
    lead, types, arrs, parts = _triple(d, L, R, P)
    return _mmchecker("plo_mmchecker_quad", lead + [bitsize, seed, batch], types + [C.c_int, C.c_uint64, C.c_int], arrs, parts)


def orbiter_quad(d, L, R, P, measure=MEASURE_NNZ, mode=MODE_PHILOX, seed=0, loops=100):
    """plo_orbiter_quad: Orbiter over Q(sqrt d) on pairs as in mmchecker_quad.  Returns (Lj, Rg, hP, report dict), each output a pair."""
    return _orbiter(d, L, R, P, measure, mode, seed, loops)


def orbiter_progress_quad(d, L, R, P, measure=MEASURE_NNZ, mode=MODE_PHILOX, seed=0, loops=100, capacity=256):
    """plo_orbiter_progress_quad: the '# Found opt:' records over Q(sqrt d), in increasing index order."""
    return _orbiter_progress(d, L, R, P, measure, mode, seed, loops, capacity)


def slp_to_csr(text, outchar="o"):
    """SLP text -> (rows, cols, ptr, col, num, den): matrixBuilder on the host (no GPU needed)."""
    h = C.c_void_p()
    rows, cols, nnz = C.c_int(), C.c_int(), C.c_int64()
    f = lib().plo_slp_build
    f.argtypes = [C.c_char_p, C.c_char, C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int64)]
    _check(f(text.encode(), outchar.encode(), C.byref(h), C.byref(rows), C.byref(cols), C.byref(nnz)))
    ptr = np.zeros(rows.value + 1, dtype=np.int64); col = np.zeros(nnz.value, dtype=np.int32)
    num = np.zeros(nnz.value, dtype=np.int64); den = np.ones(nnz.value, dtype=np.int64)
    g = lib().plo_slp_export
    g.argtypes = [C.c_void_p] * 5
    try:
        _check(g(h, _ptr(ptr), _ptr(col), _ptr(num), _ptr(den)))
    finally:
        lib().plo_slp_free.argtypes = [C.c_void_p]
        lib().plo_slp_free.restype = None
        lib().plo_slp_free(h)
    return rows.value, cols.value, ptr, col, num, den


# --------------------------------------------------------------------------
# Factorizer random restarts (SURVEY.md section 8 row f2)
# --------------------------------------------------------------------------
class FactorBest(C.Structure):
    _fields_ = [("nnz_alt", C.c_uint32), ("nno_alt", C.c_uint32), ("nnz_cob", C.c_uint32), ("pad_", C.c_uint32), ("index", C.c_uint64)]


def _factor_tuple(b):
    return (b.nnz_alt, b.nno_alt, b.nnz_cob, None if b.index == NO_INDEX else b.index)


def factor_sweep(p, M, k, seed, lo, hi, table=False):
    """M: r x n residues mod p.  Returns (nnz_alt, nno_alt, nnz_cob, index)[, table (hi-lo) x 3]."""
    M = np.ascontiguousarray(M, dtype=np.uint32)
    r, n = M.shape
    best = FactorBest()
    tab = np.zeros((max(hi - lo, 0), 3), dtype=np.uint32) if table else None
    f = lib().plo_factor_sweep
    f.argtypes = [C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(FactorBest), C.c_void_p]
    _check(f(p, r, n, k, _ptr(M), seed, lo, hi, C.byref(best), _ptr(tab) if table else None))
    return (_factor_tuple(best), tab) if table else _factor_tuple(best)


def factor_sweep_devices(ndev, p, M, k, seed, lo, hi):
    """plo_factor_sweep_devices: the index range split over the first ndev devices; (nnz_alt, nno_alt, nnz_cob, index)."""
    M = np.ascontiguousarray(M, dtype=np.uint32)
    r, n = M.shape
    best = FactorBest()
    f = lib().plo_factor_sweep_devices
    f.argtypes = [C.c_int, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(FactorBest)]
    _check(f(int(ndev), p, r, n, k, _ptr(M), seed, lo, hi, C.byref(best)))
    return _factor_tuple(best)


def factor_decode(r, seed, index):
    perm = np.zeros(r, dtype=np.int32)
    f = lib().plo_factor_decode
    f.argtypes = [C.c_int, C.c_uint64, C.c_uint64, C.c_void_p]
    _check(f(r, seed, index, _ptr(perm)))
    return perm


class FactorPlan:
    def __init__(self, p, M, k, seed):
        M = np.ascontiguousarray(M, dtype=np.uint32)
        r, n = M.shape
        self._h = C.c_void_p()
        f = lib().plo_factor_plan_create
        f.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_uint64]
        _check(f(C.byref(self._h), p, r, n, k, _ptr(M), seed))
        self.launches = lib().plo_factor_plan_launches(self._h)

    def run(self, lo, hi, stream=0):
        f = lib().plo_factor_plan_run
        f.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
        _check(f(self._h, lo, hi, C.c_void_p(stream)))

    def result(self, stream=0):
        best = FactorBest()
        f = lib().plo_factor_plan_result
        f.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(FactorBest)]
        _check(f(self._h, C.c_void_p(stream), C.byref(best)))
        return _factor_tuple(best)

    def close(self):
        if self._h:
            f = lib().plo_factor_plan_destroy
            f.argtypes = [C.c_void_p]
            f.restype = None
            f(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def factorizer(M, q=0, innerdim=0, loops=30, seed=0):
    """plo_factorizer: M (Fractions) -> (rc, Alt, CoB, report dict).  rc -1 = inner dimension outside [cols, rows]."""
    num, den = _numden(M)
    r, n = num.shape
    k = innerdim or n
    an = np.zeros((r, max(k, 1)), dtype=np.int64); ad = np.ones_like(an)
    cn = np.zeros((max(k, 1), n), dtype=np.int64); cd = np.ones_like(cn)
    rep = np.zeros(8, dtype=np.uint64)
    f = lib().plo_factorizer
    f.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64] + [C.c_void_p] * 5
    rc = f(q, r, n, _ptr(num), _ptr(den), innerdim, loops, seed, _ptr(an), _ptr(ad), _ptr(cn), _ptr(cd), _ptr(rep))
    if not (rc == -1 and lib().plo_last_error().startswith(b"Fail: inner dimension")):  # the reference's own -1 (:937-942) vs PLO_E_ARG
        _check(rc)
    report = dict(initial=tuple(int(v) for v in rep[:3]), final=tuple(int(v) for v in rep[3:6]),
                  index=None if int(rep[6]) == NO_INDEX else int(rep[6]), consistent=bool(rep[7]))
    return rc, _fractions(an, ad), _fractions(cn, cd), report


# --------------------------------------------------------------------------
# dependency Explore (SURVEY.md section 8 row f3)
# --------------------------------------------------------------------------
class DepHit(C.Structure):
    _fields_ = [("depth", C.c_int32), ("pos", C.c_int32), ("rows", C.c_int32 * 5), ("coefs", C.c_int32 * 5)]


def depender(M, level, maxnumcoeff=11, q=0, user=(), max_hits=1 << 20, text_cap=1 << 24):
    """plo_depender: returns dict(hits=[(depth, pos, rows, coefs)], nhits, ncand, coeffs, text)."""
    from fractions import Fraction
    num, den = _numden(M)
    r, n = num.shape
    un = np.array([Fraction(u).numerator for u in user], dtype=np.int64); ud = np.array([Fraction(u).denominator for u in user], dtype=np.int64)
    hits = (DepHit * max_hits)()
    nh, nc, tl, ncoef = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_int()
    text = C.create_string_buffer(text_cap)
    cn = np.zeros(maxnumcoeff, dtype=np.int64); cd = np.ones(maxnumcoeff, dtype=np.int64)
    f = lib().plo_depender
    f.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_void_p,
                  C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_char_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]
    rc = f(q, r, n, _ptr(num), _ptr(den), len(user), _ptr(un) if len(user) else None, _ptr(ud) if len(user) else None, maxnumcoeff, level,
           max_hits, C.cast(hits, C.c_void_p), C.byref(nh), C.byref(nc), text, text_cap, C.byref(tl), _ptr(cn), _ptr(cd), C.byref(ncoef))
    if rc == E_RANGE and nh.value > max_hits:  # more hits than room: the library reports the total, come back with room for all
        return depender(M, level, maxnumcoeff, q, user, max_hits=nh.value, text_cap=max(text_cap, 80 * nh.value))
    _check(rc)
    k = min(nh.value, max_hits)
    out = [(h.depth, h.pos, tuple(h.rows), tuple(h.coefs)) for h in hits[:k]]
    coeffs = [Fraction(int(a), int(b)) for a, b in zip(cn[:ncoef.value], cd[:ncoef.value])]
    return dict(hits=out, nhits=nh.value, ncand=nc.value, coeffs=coeffs, text=text.value.decode())


# --------------------------------------------------------------------------
# host-only passes around a sweep (SURVEY.md section 8 row f4)
# --------------------------------------------------------------------------
def _triple_pass(fname, head, L, R, P, shapes, stats_words=0):
    Ln, Ld = _numden(L); Rn, Rd = _numden(R); Pn, Pd = _numden(P)
    outs = []
    for shp in shapes:
        outs += [np.zeros(shp, dtype=np.int64), np.ones(shp, dtype=np.int64)]
    st = np.zeros(max(stats_words, 1), dtype=np.uint64)
    f = getattr(lib(), fname)
    f.argtypes = [C.c_int] * len(head) + [C.c_void_p] * (12 + (1 if stats_words else 0))
    args = list(head) + [_ptr(a) for a in (Ln, Ld, Rn, Rd, Pn, Pd)] + [_ptr(o) for o in outs] + ([_ptr(st)] if stats_words else [])
    rc = _check(f(*args), allow=(3,))
    return rc, [_fractions(outs[2 * t], outs[2 * t + 1]) for t in range(3)], [int(v) for v in st]


def negater(L, R, P, only_sign=False):
    """plo_negater: returns ((L', R', P'), stats[12])."""
    _, mats, st = _triple_pass("plo_negater", [1 if only_sign else 0, len(L), len(L[0]), len(R[0]), len(P)], L, R, P,
                               [(len(L), len(L[0])), (len(R), len(R[0])), (len(P), len(P[0]))], 12)
    return mats, st


def rotater(L, R, P, right=False):
    """plo_rotater: returns (rc, (L', R', P'))."""
    from . import hm
    m, k, n = hm.LRP2MM(L, R, P)
    r = len(L)
    shapes = [(r, m * n), (r, m * k), (n * k, r)] if right else [(r, k * n), (r, m * n), (m * k, r)]
    rc, mats, _ = _triple_pass("plo_rotater", [1 if right else 0, r, len(L[0]), len(R[0]), len(P)], L, R, P, shapes)
    return rc, mats


GROWTH_NAMES = ("Ginfinf", "Ginf2", "G2inf", "G22", "G2", "Q0", "Qkinfinf", "Q1inf2", "Qk12inf", "Qk2inf", "Q122")


def _growth_factors(d, L, R, P):
    lead, types, arrs, (La, Ra, Pa) = _triple(d, L, R, P)
    out = np.zeros(11, dtype=np.float64)
    f = lib().plo_growth_factors if d is None else lib().plo_growth_factors_quad
    f.argtypes = types + [C.c_int] * 4 + [C.c_void_p] * (len(arrs) + 1)
    _check(f(*lead, len(La), len(La[0]), len(Ra[0]), len(Pa), *(_ptr(x) for x in arrs), _ptr(out)))
    return dict(zip(GROWTH_NAMES, out.tolist()))


def growth_factors(L, R, P):
    """plo_growth_factors: dict of the eleven factors of src/growthfactor.cpp:199-229."""
    return _growth_factors(None, L, R, P)


def growth_factors_quad(d, L, R, P):
    """plo_growth_factors_quad: the eleven factors over Q(sqrt d), d > 0; L, R, P are pairs (rational part, sqrt(d) part) of
    lists of rows of Fraction."""
    return _growth_factors(d, L, R, P)
