"""``B200StretchMove`` of the reference-side binding (``tests/helpers/reference_b200_move.py``, INTEGRATION.md
section 4) without the reference installed: on a stub of the reference's ``RedBlueMove`` it keeps the reference's
constructor arguments, finds the engine through ``model.log_prob_fn.f.ctx`` and hands the state to
``propose_stretch``.  ``tests/test_gpu_integration.py`` runs ``propose_stretch`` itself on the GPU."""
import importlib.util
import os
import sys
import types

import numpy as np

HELPER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "helpers", "reference_b200_move.py")


class _RedBlueMove(object):
    def __init__(self, nsplits=2, randomize_split=True, live_dangerously=False):  # moves/red_blue.py:37-43
        self.nsplits = int(nsplits)
        self.live_dangerously = live_dangerously
        self.randomize_split = randomize_split


def _binding_on_stub(monkeypatch):
    emcee = types.ModuleType("emcee")
    emcee.moves = types.ModuleType("emcee.moves")
    emcee.moves.red_blue = types.ModuleType("emcee.moves.red_blue")
    emcee.moves.red_blue.RedBlueMove = _RedBlueMove
    for name, mod in (("emcee", emcee), ("emcee.moves", emcee.moves), ("emcee.moves.red_blue", emcee.moves.red_blue)):
        monkeypatch.setitem(sys.modules, name, mod)
    spec = importlib.util.spec_from_file_location("reference_b200_move_on_stub", HELPER)
    binding = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(binding)
    return binding


def test_b200_stretch_move_forwards_to_propose_stretch(monkeypatch):
    binding = _binding_on_stub(monkeypatch)
    assert issubclass(binding.B200StretchMove, _RedBlueMove)
    calls = []

    def fake_propose(*args):
        calls.append(args)
        return np.array([True, False, True, False])

    monkeypatch.setattr(binding, "propose_stretch", fake_propose)
    ctx = object()
    model = types.SimpleNamespace(log_prob_fn=types.SimpleNamespace(f=types.SimpleNamespace(ctx=ctx)))
    state = types.SimpleNamespace(coords=np.zeros((4, 2)), log_prob=np.zeros(4))
    for move, expect in [(binding.B200StretchMove(), (2.0, 2, True, False)),
                         (binding.B200StretchMove(a=1.5, nsplits=3, randomize_split=False, live_dangerously=True),
                          (1.5, 3, False, True))]:
        calls.clear()
        new_state, acc = move.propose(model, state)
        assert new_state is state and np.array_equal(acc, [True, False, True, False])
        (got,) = calls
        assert got[0] is ctx and got[1] is state.coords and got[2] is state.log_prob
        assert got[3:] == expect
