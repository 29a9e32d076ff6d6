"""The reference-side binding of INTEGRATION.md section 4, as a maintainer of dfm/emcee would add it
(``src/emcee/moves/b200.py``): a ``RedBlueMove`` whose ``propose`` forwards to the C ABI, and a device
log-probability usable as ``log_prob_fn``.  The shared library is bound with ctypes only -- nothing of
``emcee_b200``'s Python layer.  ``B200StretchMove`` subclasses the REFERENCE package's ``RedBlueMove`` and
exists only where ``emcee`` is importable; ``DeviceGaussian`` and ``propose_stretch`` need nothing but numpy.
Executed by ``tests/test_gpu_integration.py``."""
import ctypes as C
import os

import numpy as np

try:
    from emcee.moves.red_blue import RedBlueMove  # the reference's own base class (moves/red_blue.py:11)
except ImportError:
    RedBlueMove = None

_LIB = os.environ.get("EMCEE_B200_LIB") or os.path.join(
    os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), "emcee_b200", "libemcee_b200.so")
_lib = C.CDLL(_LIB)
_dp = C.POINTER(C.c_double)
_lib.eb_last_error.restype = C.c_char_p
_lib.eb_last_error.argtypes = [C.c_void_p]


class _EbMove(C.Structure):  # struct eb_move, include/emcee_b200.h (ABI 2)
    _fields_ = [("kind", C.c_int32), ("nsplits", C.c_int32), ("randomize_split", C.c_int32),
                ("live_dangerously", C.c_int32), ("weight", C.c_double), ("p0", C.c_double), ("p1", C.c_double),
                ("mode", C.c_int32), ("reserved", C.c_int32), ("seq_index", C.c_int64), ("cov", _dp), ("ncov", C.c_uint64)]


def _check(ctx, rc):
    if rc:
        msg = _lib.eb_last_error(ctx).decode()
        raise (RuntimeError if rc == -13 else ValueError)(msg)  # red_blue.py:64-70 / ensemble.py:476-479,550-551


class DeviceGaussian(object):
    """``log_prob_fn`` for ``EnsembleSampler(..., vectorize=True)``: evaluates on the GPU and owns the engine."""

    def __init__(self, nwalkers, icov, seed=0, device=0):
        d = icov.shape[0]
        self.ctx = C.c_void_p()
        _check(None, _lib.eb_create(device, C.c_int64(nwalkers), C.c_int64(d), C.c_uint64(seed), C.byref(self.ctx)))
        params = np.concatenate([np.zeros(d), np.ascontiguousarray(icov, dtype=np.float64).ravel()])
        _check(self.ctx, _lib.eb_model_set(self.ctx, 1, params.ctypes.data_as(_dp), C.c_size_t(params.size)))

    def __call__(self, coords):  # ensemble.py:486-487 (vectorised call)
        x = np.ascontiguousarray(coords, dtype=np.float64)
        out = np.empty(len(x))
        _check(self.ctx, _lib.eb_compute_log_prob(self.ctx, x.ctypes.data_as(_dp), C.c_size_t(len(x)),
                                                  out.ctypes.data_as(_dp)))
        return out

    def close(self):
        if self.ctx:
            _lib.eb_destroy(self.ctx)
            self.ctx = C.c_void_p()


def propose_stretch(ctx, coords, log_prob, a=2.0, nsplits=2, randomize_split=True, live_dangerously=False):
    """One stretch-move step of every walker on the engine ``ctx``.  ``coords`` [N, D] and ``log_prob`` [N]
    (C-contiguous float64) are updated in place; returns the accept mask.  The defaults are RedBlueMove's."""
    n = coords.shape[0]
    c = np.ascontiguousarray(coords)
    lp = np.ascontiguousarray(log_prob)
    _check(ctx, _lib.eb_set_state(ctx, c.ctypes.data_as(_dp), lp.ctypes.data_as(_dp)))
    mv = _EbMove(0, nsplits, int(randomize_split), int(live_dangerously), 1.0, a, np.nan, 0, 0, 0, None, 0)
    acc = np.zeros(n, dtype=np.uint8)
    _check(ctx, _lib.eb_step(ctx, C.byref(mv), C.c_size_t(1), C.c_uint64(1), acc.ctypes.data_as(C.POINTER(C.c_uint8))))
    _check(ctx, _lib.eb_get_state(ctx, coords.ctypes.data_as(_dp), log_prob.ctypes.data_as(_dp)))
    return acc.astype(bool)


if RedBlueMove is not None:

    class B200StretchMove(RedBlueMove):
        def __init__(self, a=2.0, **kwargs):
            self.a = a
            super(B200StretchMove, self).__init__(**kwargs)

        def propose(self, model, state):  # moves/red_blue.py:52
            ctx = model.log_prob_fn.f.ctx  # _FunctionWrapper.f, ensemble.py:633
            acc = propose_stretch(ctx, state.coords, state.log_prob, self.a, self.nsplits, self.randomize_split,
                                  self.live_dangerously)
            return state, acc
