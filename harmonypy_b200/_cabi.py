"""ctypes binding of libharmony_b200.so (include/harmony_b200.h).

There is deliberately no fallback: if the CUDA library has not been built, importing the
engine raises with the build command.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libharmony_b200.so")

# enum hmy_matrix
Z_CORR, Z_COS, Z_ORIG, R, Y, O, E, W = range(8)

ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p)

SYMBOLS = {
    "hmy_version": (C.c_char_p, []),
    "hmy_last_error": (C.c_char_p, [C.c_void_p]),
    "hmy_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int,
                             C.c_int, C.POINTER(C.c_int32)]),
    "hmy_destroy": (None, [C.c_void_p]),
    "hmy_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hmy_set_params": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float,
                                 C.c_double]),
    "hmy_set_data": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "hmy_init_from_centroids": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_double)]),
    "hmy_kmeans_init": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int, C.c_double, C.c_void_p, C.POINTER(C.c_double)]),
    "hmy_kmeans_round": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_double)]),
    "hmy_queue_perm": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hmy_objectives": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double)]),
    "hmy_host_alloc": (C.c_void_p, [C.c_int, C.c_size_t]),
    "hmy_host_free": (None, [C.c_void_p]),
    "hmy_ridge_correct": (C.c_int, [C.c_void_p]),
    "hmy_get": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]),
    "hmy_synchronize": (C.c_int, [C.c_void_p]),
    "hmy_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "hmy_counter": (C.c_int64, [C.c_void_p, C.c_char_p]),
    "hmy_timer_ms": (C.c_double, [C.c_void_p, C.c_char_p]),
    "hmy_set_allreduce": (C.c_int, [C.c_void_p, ALLREDUCE_FN, C.c_void_p]),
    "hmy_set_rank": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "hmy_comm_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hmy_comm_attach": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "hmy_lisi_compute": (C.c_int, [C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_void_p]),
}

_lib = None


class EngineError(RuntimeError):
    pass


def load():
    """Load the shared library (once) and declare every prototype of the header."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EngineError(
            f"{LIB_PATH} is missing: build it with `python -m harmonypy_b200.build` "
            "(needs nvcc; there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError here means header and library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _pinned_alloc(device, nbytes):
    """Address of `nbytes` of page-locked host memory, or None (no GPU / allocation refused)."""
    p = load().hmy_host_alloc(int(device), int(nbytes))
    return int(p) if p else None


def _pinned_free(ptr):
    load().hmy_host_free(C.c_void_p(ptr))


def _wrap_address(ptr, nbytes):
    """uint8 array over foreign memory; views taken from it keep it alive through their `base`."""
    return np.ctypeslib.as_array((C.c_ubyte * nbytes).from_address(ptr))


def pinned_empty(shape, dtype=np.float32, device=0):
    """An uninitialised array in page-locked host memory (hmy_host_alloc): hmy_set_data / hmy_get move such arrays with
    one DMA instead of staging them through bounce buffers.  The memory is released when the last view of it dies.
    Falls back to np.empty when page-locked memory is not available."""
    import weakref
    shape = tuple(int(x) for x in np.atleast_1d(shape))
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    ptr = _pinned_alloc(device, nbytes) if nbytes else None
    if ptr is None:
        return np.empty(shape, dtype=dtype)
    raw = (C.c_ubyte * nbytes).from_address(ptr)
    fin = weakref.finalize(raw, _pinned_free, ptr)        # every view's base chain ends at `raw`
    fin.atexit = False                                    # at interpreter exit the process's memory goes anyway: no CUDA calls during teardown
    return np.ctypeslib.as_array(raw).view(dtype).reshape(shape)


class _ResultPool:
    """Host buffers for the large result reads (Z_corr, R ...).  A fresh NumPy array costs one page fault per 4 KB on
    its first write -- measured: 20-40 ms of a 200 MB read-back -- so buffers whose arrays have been dropped are handed
    out again; they are page-locked when the runtime grants it, so that hmy_get fills them with one DMA (no bounce
    buffer, no host copy).  A buffer is free when nothing but the pool refers to it (the arrays returned to callers
    are views whose `base` is the buffer, so it cannot be reused while any of them -- or a slice of them -- is alive).
    Pool buffers live as long as the process (at most MAX_PER_SIZE per size)."""
    MAX_PER_SIZE = 3
    MIN_BYTES = 8 << 20

    def __init__(self):
        self._bufs = {}

    def array(self, shape, dtype, device=0):
        import sys
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        if nbytes < self.MIN_BYTES:
            return np.empty(shape, dtype=dtype)
        lst = self._bufs.setdefault(nbytes, [])
        owner = None
        for b in lst:
            if sys.getrefcount(b) == 3:          # the list, the loop variable, getrefcount's argument: no view alive
                owner = b
                break
        if owner is None:
            if len(lst) < self.MAX_PER_SIZE:
                ptr = _pinned_alloc(device, nbytes)
                owner = _wrap_address(ptr, nbytes) if ptr is not None else np.empty(nbytes, dtype=np.uint8)
                lst.append(owner)
            else:
                owner = np.empty(nbytes, dtype=np.uint8)
        return owner.view(dtype).reshape(shape)


_POOL = _ResultPool()


class Engine:
    """Thin object wrapper over one hmy_ctx (one GPU / one rank)."""

    def __init__(self, device, n_local, n_global, cell_offset, d, K, levels_per_var):
        self.lib = load()
        self.device = int(device)
        self.n_local, self.n_global, self.cell_offset = int(n_local), int(n_global), int(cell_offset)
        self.d, self.K = int(d), int(K)
        self.levels = np.ascontiguousarray(levels_per_var, dtype=np.int32)
        self.V, self.B = len(self.levels), int(self.levels.sum())
        h = C.c_void_p()
        rc = self.lib.hmy_create(C.byref(h), int(device), self.n_local, self.n_global, self.cell_offset,
                                 self.d, self.K, self.V, self.levels.ctypes.data_as(C.POINTER(C.c_int32)))
        if rc:
            raise EngineError("hmy_create: " + (self.lib.hmy_last_error(None) or b"?").decode())
        self.h = h
        self._cb = None

    def _ck(self, rc, what):
        if rc:
            raise EngineError(f"{what}: " + (self.lib.hmy_last_error(self.h) or b"?").decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.hmy_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, stream_ptr):
        self._ck(self.lib.hmy_set_stream(self.h, C.c_void_p(stream_ptr)), "hmy_set_stream")

    def set_params(self, Pr_b, theta, sigma, lamb, lambda_estimation, alpha, block_size):
        Pr_b = np.ascontiguousarray(Pr_b, dtype=np.float32)
        theta = np.ascontiguousarray(theta, dtype=np.float32)
        sigma = np.ascontiguousarray(sigma, dtype=np.float32)
        assert Pr_b.shape == (self.B,) and theta.shape == (self.B,) and sigma.shape == (self.K,)
        if lambda_estimation:
            lamb_p = None
        else:
            lamb = np.ascontiguousarray(lamb, dtype=np.float32)
            assert lamb.shape == (self.B + 1,), "lamb must have one entry per level plus the intercept"
            lamb_p = _ptr(lamb)
        self._ck(self.lib.hmy_set_params(self.h, _ptr(Pr_b), _ptr(theta), _ptr(sigma), lamb_p,
                                         int(bool(lambda_estimation)), float(alpha), float(block_size)),
                 "hmy_set_params")

    def set_data(self, Z_nxd, codes_vxn):
        Z = np.ascontiguousarray(Z_nxd, dtype=np.float32)
        codes = np.ascontiguousarray(codes_vxn, dtype=np.int32)
        assert Z.shape == (self.n_local, self.d), (Z.shape, self.n_local, self.d)
        assert codes.shape == (self.V, self.n_local)
        self._ck(self.lib.hmy_set_data(self.h, _ptr(Z), _ptr(codes)), "hmy_set_data")

    def init_from_centroids(self, Y0_kxd):
        Y0 = np.ascontiguousarray(Y0_kxd, dtype=np.float32)
        assert Y0.shape == (self.K, self.d)
        obj = (C.c_double * 3)()
        self._ck(self.lib.hmy_init_from_centroids(self.h, _ptr(Y0), obj), "hmy_init_from_centroids")
        return obj[0], obj[1], obj[2]

    def kmeans_init(self, seed, max_iter=25, tol=1e-4):
        """k-means++ / Lloyd on the resident Z_cos (hmy_kmeans_init).  Returns (K x d means, info dict).
        On a shard of the cells (n_local < n_global) it is collective: every rank calls it with the same arguments,
        after set_allreduce and set_rank, and every rank gets the same result."""
        Y = np.empty((self.K, self.d), dtype=np.float32)
        info = (C.c_double * 3)()
        self._ck(self.lib.hmy_kmeans_init(self.h, C.c_uint64(int(seed) & (2**64 - 1)), int(max_iter), float(tol), _ptr(Y), info),
                 "hmy_kmeans_init")
        return Y, {"iterations": int(info[0]), "inertia": float(info[1]), "last_shift2": float(info[2])}

    def kmeans_round(self, perm=None, wait=True):
        """One round.  wait=False (lookahead contexts): enqueue it and return None; read the sums with objectives()."""
        obj = (C.c_double * 3)() if wait else None
        if perm is None:
            p = None
        else:
            perm = np.ascontiguousarray(perm, dtype=np.int64)
            assert perm.shape == (self.n_global,)
            p = _ptr(perm)
        self._ck(self.lib.hmy_kmeans_round(self.h, p, obj), "hmy_kmeans_round")
        return (obj[0], obj[1], obj[2]) if wait else None

    def objectives(self, n):
        """Objective sums of the last n stages, oldest first (waits for the stream once)."""
        out = (C.c_double * (3 * n))()
        self._ck(self.lib.hmy_objectives(self.h, int(n), out), "hmy_objectives")
        return [(out[3 * i], out[3 * i + 1], out[3 * i + 2]) for i in range(n)]

    @property
    def lookahead(self):
        """True when the context runs the block permutations one round ahead (tensor-memory round kernel): the
        first round's permutation is queued before init, every round call carries the NEXT round's."""
        return self.counter("lookahead") == 1

    def queue_perm(self, perm=None):
        if perm is None:
            p = None
        else:
            perm = np.ascontiguousarray(perm, dtype=np.int64)
            assert perm.shape == (self.n_global,)
            p = _ptr(perm)
        self._ck(self.lib.hmy_queue_perm(self.h, p), "hmy_queue_perm")

    def ridge_correct(self):
        self._ck(self.lib.hmy_ridge_correct(self.h), "hmy_ridge_correct")

    def get(self, which):
        n, d, K, B = self.n_local, self.d, self.K, self.B
        shape, dt = {
            Z_CORR: ((n, d), np.float32), Z_COS: ((n, d), np.float32), Z_ORIG: ((n, d), np.float32),
            R: ((n, K), np.float32), Y: ((K, d), np.float32), O: ((K, B), np.float64), E: ((K, B), np.float64),
            W: ((B, K, d), np.float32),
        }[which]
        out = _POOL.array(shape, dt, self.device)
        self._ck(self.lib.hmy_get(self.h, int(which), _ptr(out), out.nbytes), "hmy_get")
        return out

    def synchronize(self):
        self._ck(self.lib.hmy_synchronize(self.h), "hmy_synchronize")

    def set_option(self, name, value):
        self._ck(self.lib.hmy_set_option(self.h, name.encode(), int(value)), f"hmy_set_option({name})")

    def counter(self, name):
        return int(self.lib.hmy_counter(self.h, name.encode()))

    def timer_ms(self, name):
        return float(self.lib.hmy_timer_ms(self.h, name.encode()))

    def comm_export(self):
        """64-byte IPC handle of this rank's exchange buffer (fused multi-GPU mode)."""
        buf = C.create_string_buffer(64)
        self._ck(self.lib.hmy_comm_export(self.h, buf), "hmy_comm_export")
        return buf.raw

    def comm_attach(self, rank, world, handles):
        """handles: the world x 64 bytes of every rank's comm_export(), in rank order."""
        blob = b"".join(handles)
        assert len(blob) == 64 * world
        self._ck(self.lib.hmy_comm_attach(self.h, int(rank), int(world), blob), "hmy_comm_attach")

    def set_rank(self, rank, world):
        """This rank's place among `world` ranks (hmy_set_rank): needed by kmeans_init on a shard of the cells."""
        self._ck(self.lib.hmy_set_rank(self.h, int(rank), int(world)), "hmy_set_rank")

    def set_allreduce(self, pyfunc):
        """pyfunc(dev_ptr:int, count:int, dtype:int, stream:int) -> 0 on success."""
        def tramp(user, ptr, count, dtype, stream):
            try:
                return int(pyfunc(ptr or 0, count, dtype, stream or 0) or 0)
            except Exception as exc:        # never let an exception cross the C boundary
                import traceback
                traceback.print_exc()
                return 1
        self._cb = ALLREDUCE_FN(tramp)      # keep alive
        self._ck(self.lib.hmy_set_allreduce(self.h, self._cb, None), "hmy_set_allreduce")
