#!/usr/bin/env python
"""Generate ``tests/golden/*.npz`` from the UNMODIFIED reference (TEST INFRASTRUCTURE).

Run in the authoring container only (``/root/reference`` does not exist on the
GPU box):

    python -m oracle.gen_golden                  # every case
    python -m oracle.gen_golden integration      # one case (or several, by name)

What it does: imports dfm/emcee from ``/root/reference/src`` (stubbing the
setuptools_scm-generated ``emcee.emcee_version`` module that
``src/emcee/__init__.py:22`` imports), builds an ``emcee.EnsembleSampler`` with
the reference's own moves, replaces ``sampler._random`` (``ensemble.py:166``) by
``oracle.philox.PhiloxRandom`` and steps it with ``sampler.sample(...)``.  Every
array written is produced by the reference's arithmetic; nothing from
``oracle/redblue.py`` or ``emcee_b200`` is involved.
"""

import os
import sys
import types

import numpy as np

REF_SRC = "/root/reference/src"
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def import_reference():
    stub = types.ModuleType("emcee.emcee_version")
    stub.__version__ = "0+reference.8ab6c0f"
    sys.modules["emcee.emcee_version"] = stub
    sys.path.insert(0, REF_SRC)
    import emcee  # noqa

    assert emcee.__file__.startswith(REF_SRC), emcee.__file__
    return emcee


def case_list(emcee):
    from . import targets as T

    mv = emcee.moves
    iso5 = T.GaussIso(5)
    rng = np.random.default_rng(777)

    def p0(n, d, scale=1.0, shift=0.0):
        return shift + scale * rng.standard_normal((n, d))

    d8 = T.make_config("gauss_dense", 64, 8)[0]
    d16 = T.make_config("gauss_dense", 96, 16)[0]
    d16m = T.GaussDense(d16.icov, mean=np.linspace(-1.0, 1.0, 16))
    return [
        # name, nwalkers, ndim, target, moves, p0, nsteps
        ("stretch_iso_32x5", 32, 5, iso5, mv.StretchMove(), p0(32, 5), 60),
        ("stretch_iso_fixedsplit_32x5", 32, 5, iso5,
         mv.StretchMove(randomize_split=False), p0(32, 5), 30),
        ("stretch_iso_a3_nsplits5_32x1", 32, 1, T.GaussIso(1),
         mv.StretchMove(a=3.0, nsplits=5), p0(32, 1), 40),
        ("stretch_iso_odd_37x3", 37, 3, T.GaussIso(3), mv.StretchMove(nsplits=3), p0(37, 3), 30),
        ("stretch_dense_64x8", 64, 8, d8, mv.StretchMove(), p0(64, 8), 40),
        ("stretch_dense_mean_96x16", 96, 16, d16m, mv.StretchMove(), p0(96, 16), 30),
        ("stretch_ring_80x6", 80, 6, T.Ring(6), mv.StretchMove(), p0(80, 6, 5.0 / np.sqrt(6)), 40),
        ("stretch_rosen_40x4", 40, 4, T.Rosenbrock(4), mv.StretchMove(), p0(40, 4, 0.1, 1.0), 40),
        ("de_rosen_40x4", 40, 4, T.Rosenbrock(4), mv.DEMove(), p0(40, 4, 0.1, 1.0), 40),
        ("de_gamma1_iso_32x5", 32, 5, iso5, mv.DEMove(sigma=1e-2, gamma0=1.0), p0(32, 5), 30),
        ("snooker_iso_40x4", 40, 4, T.GaussIso(4), mv.DESnookerMove(), p0(40, 4), 40),
        ("mix_de_snooker_rosen_48x6", 48, 6, T.Rosenbrock(6),
         [(mv.DEMove(), 0.8), (mv.DESnookerMove(), 0.2)], p0(48, 6, 0.1, 1.0), 60),
        ("mix3_ring_64x4", 64, 4, T.Ring(4),
         [(mv.StretchMove(), 0.5), (mv.DEMove(), 0.3), (mv.DESnookerMove(gammas=1.2), 0.2)],
         p0(64, 4, 2.5), 50),
        # ---- round 2: WalkMove (walk.py:27-37) and GaussianMove / MHMove (gaussian.py, mh.py:35-65) ----
        ("walk_all_rosen_40x4", 40, 4, T.Rosenbrock(4), mv.WalkMove(), p0(40, 4, 0.1, 1.0), 40),
        ("walk_s6_iso_32x5", 32, 5, iso5, mv.WalkMove(s=6), p0(32, 5), 40),
        ("walk_s3_nsplits3_ring_48x4", 48, 4, T.Ring(4), mv.WalkMove(s=3, nsplits=3), p0(48, 4, 2.5), 30),
        ("walk_all_dense_64x8", 64, 8, d8, mv.WalkMove(), p0(64, 8), 30),
        ("gauss_iso_vector_32x5", 32, 5, iso5, mv.GaussianMove(0.3), p0(32, 5), 40),
        ("gauss_iso_random_factor_rosen_40x4", 40, 4, T.Rosenbrock(4),
         mv.GaussianMove(0.05, mode="random", factor=2.0), p0(40, 4, 0.1, 1.0), 40),
        ("gauss_diag_sequential_32x5", 32, 5, iso5,
         mv.GaussianMove(np.array([0.1, 0.2, 0.3, 0.4, 0.5]), mode="sequential"), p0(32, 5), 40),
        ("gauss_full_factor_dense_64x8", 64, 8, d8,
         mv.GaussianMove(0.05 * np.linalg.inv(d8.icov), factor=1.5), p0(64, 8), 40),
        ("mix_walk_stretch_gauss_ring_64x4", 64, 4, T.Ring(4),
         [(mv.WalkMove(s=8), 0.4), (mv.StretchMove(), 0.3), (mv.GaussianMove(0.1), 0.2), (mv.WalkMove(), 0.1)],
         p0(64, 4, 2.5), 50),
    ]


def describe_moves(moves):
    """Serialise the move schedule as plain arrays: one row per move
    (kind, weight, nsplits, randomize, p0, p1) with kind 0..4 =
    stretch/de/snooker/walk/gaussian; p0,p1 = (a,-) / (sigma, gamma0 or nan) / (gammas,-) /
    (s or nan,-) / (mode 0 vector 1 random 2 sequential, factor or nan).  A GaussianMove's ``cov``
    argument (scalar, vector or matrix, as given) goes to the extra array ``move<k>_cov``."""
    if not isinstance(moves, list):
        moves = [(moves, 1.0)]
    rows, extra = [], {}
    for k, (m, w) in enumerate(moves):
        name = type(m).__name__
        if name == "StretchMove":
            rows.append([0, w, m.nsplits, m.randomize_split, m.a, np.nan])
        elif name == "DEMove":
            g = np.nan if m.gamma0 is None else m.gamma0
            rows.append([1, w, m.nsplits, m.randomize_split, m.sigma, g])
        elif name == "DESnookerMove":
            rows.append([2, w, m.nsplits, m.randomize_split, m.gammas, np.nan])
        elif name == "WalkMove":
            rows.append([3, w, m.nsplits, m.randomize_split, np.nan if m.s is None else m.s, np.nan])
        elif name == "GaussianMove":
            prop = m.get_proposal  # gaussian.py:72-119
            form = type(prop).__name__
            mode = {"vector": 0, "random": 1, "sequential": 2}[prop.mode]
            factor = np.nan if prop._log_factor is None else float(np.exp(prop._log_factor))
            rows.append([4, w, 1, 0, mode, factor])
            # recover the user's ``cov`` argument: the proposal objects keep sqrt(cov) (:45,:58) or the matrix (:50)
            extra["move%d_cov" % k] = np.asarray(prop.scale if form == "_proposal" else np.asarray(prop.scale) ** 2,
                                                 dtype=np.float64)
        else:
            raise ValueError(name)
    return np.array(rows, dtype=np.float64), extra


def model_arrays(target):
    out = {"model_kind": np.array(target.kind)}
    if target.kind == "gauss_dense":
        out["model_icov"] = target.icov
        out["model_mean"] = target.mean
    elif target.kind == "rosenbrock":
        out["model_params"] = np.array([target.a, target.b])
    elif target.kind == "ring":
        out["model_params"] = np.array([target.radius, target.sigma])
    return out


def run_case(emcee, name, nwalkers, ndim, target, moves, p0, nsteps, seed):
    from .philox import PhiloxRandom

    sampler = emcee.EnsembleSampler(nwalkers, ndim, target, moves=moves, vectorize=True)
    shim = PhiloxRandom(seed)
    shim.trace = []
    sampler._random = shim  # ensemble.py:166 -- the one injection point
    chain = np.empty((nsteps, nwalkers, ndim))
    lps = np.empty((nsteps, nwalkers))
    acc = np.empty((nsteps, nwalkers), dtype=bool)
    prev = np.zeros(nwalkers)
    k = 0
    for state in sampler.sample(p0, iterations=nsteps, skip_initial_state_check=True):
        chain[k] = state.coords
        lps[k] = state.log_prob
        now = sampler.backend.accepted.copy()
        acc[k] = (now - prev) > 0.5
        prev = now
        k += 1
    assert k == nsteps and np.array_equal(chain, sampler.get_chain())
    # draw trace of the first 3 steps, flattened per kind in call order
    tr = {}
    for kind, step, split, payload in shim.trace:
        if step is None or step >= 3:
            continue
        tr.setdefault(kind, []).append(np.atleast_1d(np.asarray(payload)).ravel())
    arrays = {
        "nwalkers": np.array(nwalkers),
        "ndim": np.array(ndim),
        "seed": np.array(seed, dtype=np.uint64),
        "moves": describe_moves(moves)[0],
        "p0": p0,
        "lp0": np.asarray(target(p0), dtype=np.float64),
        "chain": chain,
        "log_prob": lps,
        "accepted": acc,
    }
    arrays.update(describe_moves(moves)[1])
    arrays.update(model_arrays(target))
    for kind, parts in tr.items():
        arrays["trace_" + kind] = np.concatenate(parts)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrays)
    print(
        "%-32s steps=%3d  acc=%.3f  bytes=%d"
        % (name, nsteps, acc.mean(), os.path.getsize(os.path.join(OUT, name + ".npz")))
    )


INTEGRATION = os.path.join(OUT, "integration", "stretch_dense_512x16.npz")


def integration_case(emcee):
    """What ``tests/test_gpu_integration.py`` checks the engine against: the reference's own
    ``EnsembleSampler.run_mcmc`` loop and ``Backend`` with its own ``StretchMove`` (``vectorize=True``),
    512 walkers of the 16-D dense Gaussian, 25 steps, Philox key 0x1B200.  The full chain (1.6 MB) is
    not stored: per step the SHA-256 of the chain's bytes, plus the chain of a fixed sample of 32
    walkers, every log-probability and the per-walker acceptance counts."""
    import hashlib

    from . import targets as T
    from .philox import PhiloxRandom

    N, D, steps, seed = 512, 16, 25, 0x1B200
    target, p0 = T.make_config("gauss_dense", N, D)
    sampler = emcee.EnsembleSampler(N, D, target, moves=emcee.moves.StretchMove(), vectorize=True)
    sampler._random = PhiloxRandom(seed)  # ensemble.py:166
    sampler.run_mcmc(p0, steps, skip_initial_state_check=True)
    chain = sampler.get_chain()
    walkers = np.sort(np.random.default_rng(0x1B200).choice(N, 32, replace=False))
    os.makedirs(os.path.dirname(INTEGRATION), exist_ok=True)
    np.savez_compressed(
        INTEGRATION,
        seed=np.array(seed, dtype=np.uint64), icov=target.icov, p0=p0, lp0=np.asarray(target(p0)),
        chain_sha256=np.array([hashlib.sha256(np.ascontiguousarray(c).tobytes()).hexdigest() for c in chain]),
        walkers=walkers, chain_walkers=chain[:, walkers], log_prob=sampler.get_log_prob(),
        accepted=sampler.backend.accepted, acceptance_fraction=sampler.acceptance_fraction,
    )
    print("%-32s steps=%3d  acc=%.3f  bytes=%d" % (
        "integration/" + os.path.basename(INTEGRATION), steps, sampler.acceptance_fraction.mean(),
        os.path.getsize(INTEGRATION)))


def philox_kat():
    """Known answers for Philox4x32-10 itself.  The three Random123 vectors
    (kat_vectors, philox4x32-10 rows) are typed in here, not computed."""
    kat = np.array(
        [
            # ctr[4], key[2], expected[4]
            [0, 0, 0, 0, 0, 0, 0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8],
            [0xFFFFFFFF] * 6 + [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD],
            [0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344, 0xA4093822, 0x299F31D0,
             0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1],
        ],
        dtype=np.uint64,
    )
    np.save(os.path.join(OUT, "philox_kat.npy"), kat)


def main():
    os.makedirs(OUT, exist_ok=True)
    emcee = import_reference()
    philox_kat()
    only = set(sys.argv[1:])
    for idx, case in enumerate(case_list(emcee)):
        if only and case[0] not in only:
            continue
        run_case(emcee, *case, seed=0x656D636565B200 + idx)
    if not only or "integration" in only:
        integration_case(emcee)


if __name__ == "__main__":
    main()
