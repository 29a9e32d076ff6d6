"""ctypes binding of the C ABI in ``include/emcee_b200.h``.

The shared library ``libemcee_b200.so`` is built in-tree by
``__graft_entry__.build()`` (or ``make -C emcee_b200/csrc``).  There is no
fallback: if the library is missing, or no CUDA device is visible when an
engine is created, the caller gets an exception.
"""

import ctypes as C
import os

import numpy as np

__all__ = ["lib", "Engine", "EngineError", "device_count", "LIB_PATH", "EbMove"]

HERE = os.path.dirname(os.path.abspath(__file__))
# EMCEE_B200_LIB: developer override (A/B of two builds); the product always loads the in-tree library
LIB_PATH = os.environ.get("EMCEE_B200_LIB") or os.path.join(HERE, "libemcee_b200.so")

EB_OK = 0
EB_ERR_INVALID = -1
EB_ERR_CUDA = -2
EB_ERR_COMM = -3
EB_ERR_STATE = -4
EB_ERR_UNSUPPORTED = -5
EB_ERR_NAN_LOGPROB = -10
EB_ERR_INF_PARAM = -11
EB_ERR_NAN_PARAM = -12
EB_ERR_FEW_WALKERS = -13
EB_ERR_NAN_INITIAL = -14

EB_LAUNCH_CONFIG_FIELDS = 8
LAUNCH_KERNELS = ("none", "generic", "tma_rows", "dense_dmma")

EB_COMM_ID_BYTES = 128
EB_IPC_BLOB_BYTES = 256
EB_COMM_ALLGATHER = 0
EB_COMM_P2P = 1

MODEL_KINDS = {"gauss_iso": 0, "gauss_dense": 1, "rosenbrock": 2, "ring": 3}
MOVE_KINDS = {"stretch": 0, "de": 1, "snooker": 2, "walk": 3, "gaussian": 4}


class EbMove(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("nsplits", C.c_int32),
        ("randomize_split", C.c_int32),
        ("live_dangerously", C.c_int32),
        ("weight", C.c_double),
        ("p0", C.c_double),
        ("p1", C.c_double),
        # ABI 2: GaussianMove
        ("mode", C.c_int32),
        ("reserved", C.c_int32),
        ("seq_index", C.c_int64),
        ("cov", C.POINTER(C.c_double)),
        ("ncov", C.c_uint64),
    ]


class EngineError(RuntimeError):
    """A failing C-ABI call that does not map onto one of the reference's own
    exception types."""


_dp = C.POINTER(C.c_double)
_SIGNATURES = {
    "eb_abi_version": (C.c_int, []),
    "eb_device_count": (C.c_int, []),
    "eb_create": (C.c_int, [C.c_int, C.c_int64, C.c_int64, C.c_uint64, C.POINTER(C.c_void_p)]),
    "eb_destroy": (C.c_int, [C.c_void_p]),
    "eb_last_error": (C.c_char_p, [C.c_void_p]),
    "eb_model_set": (C.c_int, [C.c_void_p, C.c_int, _dp, C.c_size_t]),
    "eb_set_state": (C.c_int, [C.c_void_p, _dp, _dp]),
    "eb_get_state": (C.c_int, [C.c_void_p, _dp, _dp]),
    "eb_owned_rows": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "eb_get_state_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _dp, _dp]),
    "eb_compute_log_prob": (C.c_int, [C.c_void_p, _dp, C.c_size_t, _dp]),
    "eb_set_rng": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64]),
    "eb_get_rng": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "eb_step": (C.c_int, [C.c_void_p, C.POINTER(EbMove), C.c_size_t, C.c_uint64, C.POINTER(C.c_uint8)]),
    "eb_step_store": (
        C.c_int,
        [C.c_void_p, C.POINTER(EbMove), C.c_size_t, C.c_uint64, C.c_uint64, _dp, _dp, _dp],
    ),
    "eb_get_naccepted": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "eb_reset_counters": (C.c_int, [C.c_void_p]),
    "eb_move_picks": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.c_size_t]),
    "eb_moments": (C.c_int, [C.c_void_p, _dp, _dp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "eb_walkers_gram": (C.c_int, [C.c_void_p, _dp, C.c_size_t, _dp, C.POINTER(C.c_int)]),
    "eb_autocorr": (C.c_int, [C.c_void_p, _dp, C.c_size_t, C.c_size_t, C.c_size_t, _dp]),
    "eb_last_step_timing": (C.c_int, [C.c_void_p, _dp, C.POINTER(C.c_uint64)]),
    "eb_debug_taps": (
        C.c_int,
        [C.c_void_p, C.POINTER(C.c_int64), _dp, _dp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)],
    ),
    "eb_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "eb_debug_timeline": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.c_size_t, C.POINTER(C.c_size_t)]),
    "eb_debug_launch_config": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.c_size_t]),
    "eb_last_kernel_name": (C.c_char_p, [C.c_void_p]),
    "eb_microbench": (C.c_int, [C.c_int, C.c_int, _dp]),
    "eb_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "eb_host_free": (C.c_int, [C.c_void_p]),
    "eb_comm_id": (C.c_int, [C.c_char_p]),
    "eb_comm_init": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int]),
    "eb_comm_export": (C.c_int, [C.c_void_p, C.c_char_p]),
    "eb_comm_import": (C.c_int, [C.c_void_p, C.c_char_p]),
    "eb_comm_probe": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp]),
}

_lib = None


def lib():
    """The loaded shared library (loaded once; raises if it was not built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "emcee_b200: %s is missing -- build it with `python -c 'import "
                "__graft_entry__ as g; g.build()'` or `make -C emcee_b200/csrc`. "
                "There is no CPU fallback." % LIB_PATH
            )
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            if os.environ.get("EMCEE_B200_LIB") and not hasattr(handle, name):
                continue  # A/B against an older build
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def exported_symbols():
    return sorted(_SIGNATURES)


def device_count():
    return int(lib().eb_device_count())


def microbench(what, warps_per_sm=16):
    """TFLOP/s (what = 0 DFMA, 1..3 DMMA shapes) or GB/s (4 = HBM copy)."""
    out = C.c_double()
    rc = lib().eb_microbench(int(what), int(warps_per_sm), C.byref(out))
    if rc != EB_OK:
        raise EngineError("eb_microbench failed (%d)" % rc)
    return float(out.value)


class _PinnedOwner(object):
    def __init__(self, ptr):
        self.ptr = ptr

    def __del__(self):
        try:
            lib().eb_host_free(self.ptr)
        except Exception:
            pass


def pinned_empty(shape, dtype=np.float64):
    """numpy array in page-locked host memory (full-speed H2D / D2H)."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    ptr = C.c_void_p()
    rc = lib().eb_host_alloc(max(n, 1), C.byref(ptr))
    if rc != EB_OK:
        raise EngineError("eb_host_alloc(%d) failed" % n)
    buf = (C.c_char * max(n, 1)).from_address(ptr.value)
    buf._owner = _PinnedOwner(ptr)  # freed when the last array viewing `buf` dies
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


def _as_dp(a):
    return a.ctypes.data_as(_dp)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and a.shape != shape:
        raise ValueError("incompatible input dimensions {0}".format(a.shape))
    return a


class Engine(object):
    """Thin owner of one ``eb_ctx``.  Maps error codes onto the exception types
    the reference raises for the same conditions (``ensemble.py:314-323,
    357-358,476-479,550-551``; ``moves/red_blue.py:64-70``)."""

    def __init__(self, nwalkers, ndim, seed, device=0):
        self._h = C.c_void_p()
        self.nwalkers, self.ndim = int(nwalkers), int(ndim)
        rc = lib().eb_create(int(device), self.nwalkers, self.ndim, int(seed) & (2**64 - 1), C.byref(self._h))
        if rc != EB_OK:
            msg = lib().eb_last_error(None).decode()
            self._h = C.c_void_p()
            raise (ValueError if rc == EB_ERR_INVALID else EngineError)(msg)

    # -- plumbing -------------------------------------------------------------
    def _check(self, rc):
        if rc == EB_OK:
            return
        msg = lib().eb_last_error(self._h).decode()
        if rc in (EB_ERR_INVALID, EB_ERR_NAN_LOGPROB, EB_ERR_INF_PARAM, EB_ERR_NAN_PARAM, EB_ERR_NAN_INITIAL):
            raise ValueError(msg)
        if rc == EB_ERR_UNSUPPORTED:
            raise NotImplementedError(msg)
        if rc == EB_ERR_FEW_WALKERS:
            raise RuntimeError(msg)
        raise EngineError("%s (eb_status %d)" % (msg, rc))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().eb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- model / state ----------------------------------------------------------
    def set_model(self, kind, params):
        params = _f64(np.asarray(params, dtype=np.float64).ravel())
        self._check(lib().eb_model_set(self._h, MODEL_KINDS[kind], _as_dp(params), params.size))

    def set_state(self, coords, log_prob=None):
        coords = _f64(coords, (self.nwalkers, self.ndim))
        lp = None if log_prob is None else _f64(log_prob, (self.nwalkers,))
        self._check(lib().eb_set_state(self._h, _as_dp(coords), None if lp is None else _as_dp(lp)))

    def get_state(self, coords=None, log_prob=None):
        """Device -> host copy of the live state, into fresh arrays or into the
        given (C-contiguous float64, e.g. pinned) buffers."""
        coords = np.empty((self.nwalkers, self.ndim), dtype=np.float64) if coords is None else coords
        lp = np.empty(self.nwalkers, dtype=np.float64) if log_prob is None else log_prob
        assert coords.flags.c_contiguous and coords.dtype == np.float64 and coords.shape == (self.nwalkers, self.ndim)
        assert lp.flags.c_contiguous and lp.dtype == np.float64 and lp.shape == (self.nwalkers,)
        self._check(lib().eb_get_state(self._h, _as_dp(coords), _as_dp(lp)))
        return coords, lp

    def owned_rows(self):
        """``(row0, nrows)`` of the walkers this engine updates (all of them on one GPU)."""
        r0, n = C.c_int64(), C.c_int64()
        self._check(lib().eb_owned_rows(self._h, C.byref(r0), C.byref(n)))
        return int(r0.value), int(n.value)

    def get_state_rows(self, row0, nrows, coords, log_prob):
        """Device -> host copy of rows ``[row0, row0 + nrows)`` into the matching
        row slices of the full-size host arrays ``coords`` / ``log_prob`` (not collective)."""
        assert coords.flags.c_contiguous and coords.dtype == np.float64 and coords.shape == (self.nwalkers, self.ndim)
        assert log_prob.flags.c_contiguous and log_prob.dtype == np.float64 and log_prob.shape == (self.nwalkers,)
        c, lp = coords[row0 : row0 + nrows], log_prob[row0 : row0 + nrows]
        self._check(lib().eb_get_state_rows(self._h, int(row0), int(nrows), _as_dp(c), _as_dp(lp)))
        return coords, log_prob

    def moments(self):
        """``(mean[D], cov[D, D], count, naccepted_total)`` of the samples folded in so far
        (option ``moments_every``); per rank on a sharded ensemble."""
        mean = np.empty(self.ndim)
        cov = np.empty((self.ndim, self.ndim))
        n, na = C.c_uint64(), C.c_uint64()
        self._check(lib().eb_moments(self._h, _as_dp(mean), _as_dp(cov), C.byref(n), C.byref(na)))
        return mean, cov, int(n.value), int(na.value)

    def walkers_gram(self, coords):
        """``(gram[D, D], flags)`` of ``eb_walkers_gram`` for ``coords[rows, D]``."""
        coords = _f64(coords)
        if coords.ndim != 2 or coords.shape[1] != self.ndim:
            raise ValueError("incompatible input dimensions {0}".format(coords.shape))
        gram = np.empty((self.ndim, self.ndim))
        flags = C.c_int()
        self._check(lib().eb_walkers_gram(self._h, _as_dp(coords), coords.shape[0], _as_dp(gram), C.byref(flags)))
        return gram, int(flags.value)

    def autocorr_function(self, chain):
        """Walker-averaged normalised autocorrelation function ``[n_step, n_param]`` of
        ``chain[n_step, n_walker, n_param]`` (``eb_autocorr``)."""
        chain = _f64(chain)
        if chain.ndim != 3:
            raise ValueError("invalid dimensions")
        n_t, n_w, n_d = chain.shape
        out = np.empty((n_d, n_t), dtype=np.float64)
        self._check(lib().eb_autocorr(self._h, _as_dp(chain), n_t, n_w, n_d, _as_dp(out)))
        return np.ascontiguousarray(out.T)

    def compute_log_prob(self, coords):
        coords = _f64(coords)
        if coords.shape[-1] != self.ndim:
            raise ValueError("incompatible input dimensions {0}".format(coords.shape))
        flat = coords.reshape(-1, self.ndim)
        out = np.empty(flat.shape[0], dtype=np.float64)
        self._check(lib().eb_compute_log_prob(self._h, _as_dp(flat), flat.shape[0], _as_dp(out)))
        return out.reshape(coords.shape[:-1])

    # -- rng -----------------------------------------------------------------
    def set_rng(self, seed, step):
        self._check(lib().eb_set_rng(self._h, int(seed) & (2**64 - 1), int(step)))

    def get_rng(self):
        seed, step = C.c_uint64(), C.c_uint64()
        self._check(lib().eb_get_rng(self._h, C.byref(seed), C.byref(step)))
        return int(seed.value), int(step.value)

    # -- stepping ----------------------------------------------------------------
    @staticmethod
    def pack_moves(moves):
        """``moves``: list of (descriptor dict, weight)."""
        arr = (EbMove * len(moves))()
        for k, (d, w) in enumerate(moves):
            arr[k].kind = MOVE_KINDS[d["kind"]]
            arr[k].nsplits = int(d["nsplits"])
            arr[k].randomize_split = int(bool(d["randomize_split"]))
            arr[k].live_dangerously = int(bool(d["live_dangerously"]))
            arr[k].weight = float(w)
            arr[k].p0 = float(d["p0"])
            arr[k].p1 = float(d["p1"])
            if d.get("cov") is not None:  # GaussianMove: the array must outlive the call -> kept on `arr`
                cov = np.ascontiguousarray(d["cov"], dtype=np.float64)
                keep = getattr(arr, "_keep", [])
                keep.append(cov)
                arr._keep = keep
                arr[k].cov = cov.ctypes.data_as(_dp)
                arr[k].ncov = cov.size
                arr[k].mode = int(d.get("mode", 0))
                arr[k].seq_index = int(d.get("seq_index", 0))
        return arr

    def move_picks(self, nmoves):
        """How many steps of the last stepping call ran each schedule entry."""
        out = np.zeros(int(nmoves), dtype=np.uint64)
        self._check(lib().eb_move_picks(self._h, out.ctypes.data_as(C.POINTER(C.c_uint64)), int(nmoves)))
        return out

    def step(self, moves, nsteps, want_accepted=True):
        arr = self.pack_moves(moves)
        acc = np.zeros(self.nwalkers, dtype=np.uint8) if want_accepted else None
        self._check(
            lib().eb_step(
                self._h, arr, len(arr), int(nsteps),
                None if acc is None else acc.ctypes.data_as(C.POINTER(C.c_uint8)),
            )
        )
        return None if acc is None else acc.astype(bool)

    def step_store(self, moves, nsteps, thin_by, chain, log_prob, accepted):
        arr = self.pack_moves(moves)
        assert chain.flags.c_contiguous and log_prob.flags.c_contiguous and accepted.flags.c_contiguous
        assert chain.dtype == np.float64 and log_prob.dtype == np.float64 and accepted.dtype == np.float64
        self._check(
            lib().eb_step_store(
                self._h, arr, len(arr), int(nsteps), int(thin_by),
                _as_dp(chain), _as_dp(log_prob), _as_dp(accepted),
            )
        )

    def naccepted(self):
        out = np.zeros(self.nwalkers, dtype=np.uint64)
        self._check(lib().eb_get_naccepted(self._h, out.ctypes.data_as(C.POINTER(C.c_uint64))))
        return out

    def reset_counters(self):
        self._check(lib().eb_reset_counters(self._h))

    def last_step_timing(self):
        ms, n = C.c_double(), C.c_uint64()
        self._check(lib().eb_last_step_timing(self._h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def last_kernel_name(self):
        return lib().eb_last_kernel_name(self._h).decode()

    def set_option(self, name, value):
        self._check(lib().eb_set_option(self._h, name.encode(), int(value)))

    def debug_taps(self):
        n = self.nwalkers
        partners = np.empty((3, n), dtype=np.int64)
        scalar = np.empty(n, dtype=np.float64)
        u = np.empty(n, dtype=np.float64)
        active = np.empty(n, dtype=np.int64)
        cnt = C.c_int64()
        i64 = C.POINTER(C.c_int64)
        self._check(
            lib().eb_debug_taps(
                self._h, partners.ctypes.data_as(i64), _as_dp(scalar), _as_dp(u),
                active.ctypes.data_as(i64), C.byref(cnt),
            )
        )
        k = int(cnt.value)
        return dict(partners=partners[:, :k], scalar=scalar[:k], u_accept=u[:k], active=active[:k])

    def launch_config(self):
        """Launch shape of the last fused red-blue half-step (``eb_debug_launch_config``): kernel name,
        ``width`` (walkers per tile; lanes per walker for ``generic``), ``epl``, ``own_reg``, ``warps`` and
        ``threads`` per CTA, ``grid`` (CTAs) and ``tiles`` (active walkers for ``generic``)."""
        out = np.zeros(EB_LAUNCH_CONFIG_FIELDS, dtype=np.int64)
        self._check(lib().eb_debug_launch_config(self._h, out.ctypes.data_as(C.POINTER(C.c_int64)), out.size))
        keys = ("kernel", "width", "epl", "own_reg", "warps", "threads", "grid", "tiles")
        cfg = dict(zip(keys, (int(v) for v in out)))
        cfg["kernel"] = LAUNCH_KERNELS[cfg["kernel"]]
        return cfg

    def debug_timeline(self):
        """[SM, consumer, tile, event] cycle stamps of the last dense_dmma half-step."""
        buf = np.zeros(1 << 21, dtype=np.int64)
        n = C.c_size_t()
        self._check(lib().eb_debug_timeline(self._h, buf.ctypes.data_as(C.POINTER(C.c_int64)), buf.size, C.byref(n)))
        return buf[: n.value].reshape(-1, 8, 8, 10)  # events 0..5 consumer, 6..8 producer (dense_dmma.cu)

    # -- multi-GPU ---------------------------------------------------------------
    @staticmethod
    def comm_id():
        buf = C.create_string_buffer(EB_COMM_ID_BYTES)
        rc = lib().eb_comm_id(buf)
        if rc != EB_OK:
            raise EngineError("eb_comm_id failed (is libnccl.so.2 loadable?)")
        return buf.raw

    def comm_init(self, comm_id, rank, nranks, mode=EB_COMM_ALLGATHER):
        assert len(comm_id) == EB_COMM_ID_BYTES
        self._check(lib().eb_comm_init(self._h, comm_id, int(rank), int(nranks), int(mode)))

    def comm_export(self):
        buf = C.create_string_buffer(EB_IPC_BLOB_BYTES)
        self._check(lib().eb_comm_export(self._h, buf))
        return buf.raw

    def comm_probe(self, peer, what):
        out = C.c_double()
        self._check(lib().eb_comm_probe(self._h, int(peer), int(what), C.byref(out)))
        return float(out.value)

    def comm_import(self, blobs):
        self._check(lib().eb_comm_import(self._h, blobs))
