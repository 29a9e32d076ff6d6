"""INTEGRATION.md section 4, against the unmodified reference: ``tests/golden/integration/stretch_dense_512x16.npz``
holds what the reference's own ``EnsembleSampler.run_mcmc`` loop and ``Backend`` produced with its own StretchMove
and the Philox key below (``oracle/gen_golden.py``, ``integration_case``).  Here the engine takes that move's place
through the reference-side ctypes binding ``tests/helpers/reference_b200_move.py``, stepped the way the reference's
loop steps a move.  The chain must equal the recorded one, and the oracle's, bit for bit (stretch move)."""
import hashlib
import os
import sys

import numpy as np
import pytest

from oracle import redblue as rb
from oracle import targets as T

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "integration", "stretch_dense_512x16.npz")


def _run_like_the_reference(binding, model, p0, steps):
    """``EnsembleSampler.sample`` with one red-blue move (ensemble.py:350-351, 403-417): the initial
    log-probabilities from the vectorised ``log_prob_fn``, then per step ``propose`` and ``Backend.save_step``."""
    coords = np.array(p0, dtype=np.float64)
    log_prob = model(coords)
    log_prob0 = log_prob.copy()
    chain = np.empty((steps,) + coords.shape)
    lps = np.empty((steps, len(coords)))
    accepted = np.zeros(len(coords))
    for k in range(steps):
        accepted += binding.propose_stretch(model.ctx, coords, log_prob)
        chain[k], lps[k] = coords, log_prob
    return log_prob0, chain, lps, accepted


def test_reference_sampler_drives_the_engine():
    g = np.load(GOLDEN)
    sys.path.insert(0, os.path.join(ROOT, "tests", "helpers"))
    try:
        import reference_b200_move as binding

        (N, D), steps, seed = g["p0"].shape, len(g["chain_sha256"]), int(g["seed"])
        model = binding.DeviceGaussian(N, g["icov"], seed=seed)
        lp0, chain, lps, accepted = _run_like_the_reference(binding, model, g["p0"], steps)
        model.close()

        # the recorded run of the unmodified reference
        np.testing.assert_allclose(lp0, g["lp0"], rtol=1e-12, atol=1e-12)
        for k in range(steps):
            assert hashlib.sha256(chain[k].tobytes()).hexdigest() == g["chain_sha256"][k], k
        assert np.array_equal(chain[:, g["walkers"]], g["chain_walkers"])
        np.testing.assert_allclose(lps, g["log_prob"], rtol=1e-12, atol=1e-12)
        assert np.array_equal(accepted, g["accepted"])
        assert np.array_equal(accepted / float(steps), g["acceptance_fraction"])
        assert 0.1 < g["acceptance_fraction"].mean() < 0.9

        # and the oracle, step by step
        o = rb.OracleSampler(N, D, T.GaussDense(g["icov"]), [(rb.Stretch(), 1.0)], seed=seed)
        o.set_state(g["p0"])
        acc_total = np.zeros(N)
        for k in range(steps):
            acc_total += o.run(1)
            assert np.array_equal(chain[k], o.coords), k
        np.testing.assert_allclose(lps[-1], o.log_prob, rtol=1e-12, atol=1e-12)
        assert np.array_equal(accepted, acc_total)

        # the reference's guard still fires through the binding (red_blue.py:64-70)
        few = binding.DeviceGaussian(8, g["icov"])
        x = np.array(g["p0"][:8])
        lp = few(x)
        with pytest.raises(RuntimeError, match="fewer walkers than twice the number of dimensions"):
            binding.propose_stretch(few.ctx, x, lp)
        few.close()
    finally:
        sys.path.remove(os.path.join(ROOT, "tests", "helpers"))
