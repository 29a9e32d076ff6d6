"""CPU-side checks of the drop-in boundary: the library loads, exports every
symbol the header declares, and fails loudly without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

import emcee_b200
from emcee_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "emcee_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(eb_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    handle = ctypes.CDLL(_lib.LIB_PATH)
    names = header_symbols()
    assert len(names) >= 20
    for name in names:
        assert hasattr(handle, name), name
    # and the ctypes binding covers the whole header
    assert set(_lib.exported_symbols()) == set(names)


def test_abi_version():
    assert _lib.lib().eb_abi_version() == 2


def test_launch_config_needs_a_context_and_room_for_every_field():
    out = (ctypes.c_int64 * _lib.EB_LAUNCH_CONFIG_FIELDS)()
    assert _lib.lib().eb_debug_launch_config(None, out, len(out)) == _lib.EB_ERR_INVALID


def test_eb_move_layout_matches_header():
    # ABI 2: kind, nsplits, randomize_split, live_dangerously | weight, p0, p1 | mode, reserved | seq_index | cov* | ncov
    assert ctypes.sizeof(_lib.EbMove) == 4 * 4 + 3 * 8 + 2 * 4 + 8 + 8 + 8
    assert _lib.EbMove.cov.offset == 56 and _lib.EbMove.ncov.offset == 64


@pytest.mark.skipif(_lib.device_count() > 0, reason="only meaningful without a GPU")
def test_no_cpu_fallback():
    with pytest.raises(_lib.EngineError, match="no CPU fallback"):
        emcee_b200.EnsembleSampler(32, 5, emcee_b200.models.GaussianIso())


def test_argument_validation_needs_no_gpu():
    with pytest.raises(TypeError):
        emcee_b200.EnsembleSampler(32, 5, lambda x: 0.0)
    with pytest.raises(NotImplementedError):
        emcee_b200.EnsembleSampler(32, 5, emcee_b200.models.GaussianIso(), pool=object())
    with pytest.raises(TypeError):
        emcee_b200.models.GaussianIso()(np.zeros(5))
    with pytest.raises(ValueError):
        emcee_b200.models.GaussianDense(np.zeros((3, 4)))


def test_state_protocol():
    # reference: tests/unit/test_state.py:14-72
    s = emcee_b200.State(np.arange(6.0).reshape(3, 2), log_prob=np.zeros(3), random_state="r")
    coords, lp, rs = s
    assert len(s) == 3 and s[2] == "r" and s[-1] == "r" and np.array_equal(s[0], coords)
    with pytest.raises(IndexError):
        s[3]
    s4 = emcee_b200.State(np.zeros((3, 2)), log_prob=np.zeros(3), blobs=np.ones(3), random_state="r")
    assert len(s4) == 4 and np.array_equal(s4[3], np.ones(3)) and np.array_equal(s4[-1], np.ones(3))
    x = np.zeros((3, 2))
    c = emcee_b200.State(x, copy=True)
    c.coords += 1
    assert np.all(x == 0)
    again = emcee_b200.State(s4)
    assert again.coords is s4.coords and again.blobs is s4.blobs


def test_new_move_constructors_validate_like_the_reference():
    # reference: moves/gaussian.py:36-79, moves/mh.py:31-33, moves/walk.py:24-26
    from emcee_b200 import moves

    g = moves.GaussianMove(0.5)
    d = g.descriptor()
    assert d["kind"] == "gaussian" and d["mode"] == 0 and d["cov"].shape == (1,) and np.isnan(d["p1"])
    assert moves.GaussianMove([0.1, 0.2], mode="random", factor=2.0).descriptor()["p1"] == 2.0
    assert moves.GaussianMove(np.eye(3)).ndim == 3
    with pytest.raises(ValueError, match="not a recognized mode"):
        moves.GaussianMove(np.eye(3), mode="random")
    with pytest.raises(ValueError, match="not a recognized mode"):
        moves.GaussianMove(1.0, mode="bogus")
    with pytest.raises(ValueError, match="factor"):
        moves.GaussianMove(1.0, factor=0.5)
    with pytest.raises(ValueError, match="Invalid proposal scale dimensions"):
        moves.GaussianMove(np.zeros((2, 3)))
    with pytest.raises(NotImplementedError):
        moves.MHMove(lambda x, rng: (x, np.zeros(len(x))))
    seq = moves.GaussianMove(np.ones(4), mode="sequential")
    seq._advance(6, 4)
    assert seq.index == 2 and seq.descriptor()["seq_index"] == 2
    w = moves.WalkMove(s=7, nsplits=3)
    assert w.descriptor()["kind"] == "walk" and w.descriptor()["p0"] == 7.0 and w.descriptor()["nsplits"] == 3
    assert np.isnan(moves.WalkMove().descriptor()["p0"])


def test_move_update_host():
    # reference: moves/move.py:12-45
    from emcee_b200.moves import Move

    old = emcee_b200.State(np.zeros((4, 2)), log_prob=np.zeros(4))
    new = emcee_b200.State(np.ones((2, 2)) * [[1], [2]], log_prob=np.array([10.0, 20.0]))
    subset = np.array([True, False, True, False])
    accepted = np.array([False, False, True, False])
    Move().update(old, new, accepted, subset)
    assert np.array_equal(old.coords[2], [2, 2]) and old.log_prob[2] == 20.0 and np.all(old.coords[0] == 0)
