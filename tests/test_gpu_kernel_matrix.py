"""Every variant of the three fused half-step kernels against the oracle.

The host picks the kernel and its shape from (move, model, ndim): tma_rows with R walkers per tile
(16/8/4/2/1), the register path (EPL = 8, 8 elements per lane, when ndim == 8 * 32 / R), the own row in
registers (OWN_REG, stretch rows of at most 512 bytes) and 8..16 warps; the generic kernel with 4/8/16/32
lanes per walker; dense_dmma for stretch + gauss_dense at ndim = 8k <= 128.  Each case below names the
variant it covers and asserts it through Engine.launch_config(), so a retuned heuristic fails here instead
of silently testing something else.

Option "grid_cap" shrinks the grid of the SM-sized launches so that a few thousand walkers give every warp
(tma_rows) or consumer (dense_dmma) several tiles: the two-stage ring, its mbarrier parity flips, stage reuse
after bulk stores and -- with more than G tiles per warp -- the hand-off to the next batch of per-walker draws.

Comparisons, as in test_gpu_parity:
  * resynchronised single steps (device and oracle start from the same state and draw counter):
    accept masks bit-exact; stretch coordinates bit-exact; DE / snooker coordinates rtol = atol = 1e-12;
    log-probabilities rtol 1e-12, see _lp_tols for the two models that need an absolute term;
  * free-running steps: stretch bit-exact, the other moves within test_gpu_parity._tols.
"""
import numpy as np
import pytest

from oracle import redblue as rb
from oracle import targets as T

from gpu_util import device_model, device_moves, move_rows_from_oracle
from test_gpu_parity import _tols

import emcee_b200
from emcee_b200 import moves as dmoves

pytestmark = pytest.mark.gpu

OMOVE = {"stretch": rb.Stretch, "de": rb.DE, "snooker": rb.Snooker}
MODELS = ("gauss_iso", "ring", "rosenbrock", "gauss_dense")


def _lanes_per_walker(D):
    """the generic kernel's lanes per walker: the least power of two >= 4 with 4 lanes * 4 >= ndim, at most 32"""
    g = 4
    while g < 32 and 4 * g < D:
        g *= 2
    return g


def _lp_tols(model, D):
    """(rtol, atol) of a resynchronised step's log-probabilities."""
    if model == "rosenbrock":
        # t = x1 - x0 * x0 may be contracted into one FMA on the device; numpy rounds x0 * x0 first.  That
        # is <= 1 ulp of x0^2 per element, times 2 b |t| ~ 60 for the chains here: 2e-14 per term.
        return 1e-12, 2e-14 * D
    if model == "gauss_dense":
        # the quadratic form of the paper's precision matrix (condition number ~1e4..1e5) in a different
        # summation order, the bound test_gpu_parity uses for the dense model
        return 1e-11, 1e-11
    return 1e-12, 1e-12


class Pair(object):
    """A device engine and the oracle, on the same target, moves, seed and initial state."""

    def __init__(self, model, N, D, omoves, seed, options=(), target=None, p0=None, dmoves_=None):
        if target is None:
            target, p0 = T.make_config(model, N, D)
        self.model, self.N, self.D, self.seed = model, N, D, seed
        self.omoves = omoves
        self.o = rb.OracleSampler(N, D, target, omoves, seed=seed)
        mv = dmoves_ if dmoves_ is not None else device_moves(move_rows_from_oracle(omoves))
        s = emcee_b200.EnsembleSampler(N, D, device_model(model, target=target), moves=mv, seed=seed)
        self.eng, self.sched = s._engine, s._schedule()
        self._keep = s
        for k, v in options:
            self.eng.set_option(k, v)
        self.eng.set_state(p0)
        _, lp0 = self.eng.get_state()
        self.o.set_state(p0, lp0)  # both start from the device's log-probabilities
        self.p0, self.lp0 = p0, lp0

    def kinds(self):
        return {m.kind for m, _ in self.omoves}

    def free_run(self, nsteps, label=""):
        g = dict(moves=move_rows_from_oracle(self.omoves))
        exact, rtol, atol = _tols(g)
        lrt, lat = _lp_tols(self.model, self.D)
        for k in range(nsteps):
            acc_o = self.o.run(1)
            acc = self.eng.step(self.sched, 1)
            coords, lp = self.eng.get_state()
            assert np.array_equal(acc, acc_o), (label, "free step", k)
            if exact:
                assert np.array_equal(coords, self.o.coords), (label, "free step", k)
            else:
                np.testing.assert_allclose(coords, self.o.coords, rtol=rtol, atol=atol, err_msg="%s free %d" % (label, k))
            np.testing.assert_allclose(
                lp, self.o.log_prob, rtol=max(rtol, lrt), atol=max(10 * atol, lat), err_msg="%s free %d lp" % (label, k)
            )
        assert np.array_equal(self.eng.naccepted(), self.o.naccepted.astype(np.uint64)), label

    def single_steps(self, nsteps, label=""):
        stretch = self.kinds() == {"stretch"}
        lrt, lat = _lp_tols(self.model, self.D)
        for k in range(nsteps):
            self.eng.set_state(self.o.coords, self.o.log_prob)
            self.eng.set_rng(self.seed, self.o.step)
            acc_o = self.o.run(1)
            acc = self.eng.step(self.sched, 1)
            coords, lp = self.eng.get_state()
            assert np.array_equal(acc, acc_o), (label, "step", k)
            if stretch:
                assert np.array_equal(coords, self.o.coords), (label, "step", k)
            else:
                np.testing.assert_allclose(coords, self.o.coords, rtol=1e-12, atol=1e-12, err_msg="%s step %d" % (label, k))
            np.testing.assert_allclose(lp, self.o.log_prob, rtol=lrt, atol=lat, err_msg="%s step %d lp" % (label, k))
        assert np.array_equal(self.eng.naccepted(), self.o.naccepted.astype(np.uint64)), label


def _assert_config(cfg, kernel, width, epl=0, own_reg=0, warps=None, label=""):
    got = (cfg["kernel"], cfg["width"], cfg["epl"], cfg["own_reg"])
    assert got == (kernel, width, epl, own_reg), (label, cfg)
    if warps is not None:
        assert cfg["warps"] == warps, (label, cfg)


def test_grid_cap_and_launch_config_hooks():
    p = Pair("gauss_iso", 64, 32, [(rb.Stretch(), 1.0)], seed=1)
    assert p.eng.launch_config()["kernel"] == "none"  # nothing stepped yet
    with pytest.raises(ValueError, match="grid_cap"):
        p.eng.set_option("grid_cap", -1)
    p.eng.set_option("grid_cap", 0)
    p.free_run(1)
    cfg = p.eng.launch_config()
    assert cfg["kernel"] == "tma_rows" and cfg["threads"] == 32 * cfg["warps"] and cfg["tiles"] == 4 and cfg["grid"] == 1


# ---- tma_rows: every (move x model) x every reachable (R, EPL, OWN_REG) ------------------------------------
# (move, ndim, R, EPL, OWN_REG, warps): ndims picked from the selection rule of launch_tma_t
TMA_CELLS = [
    ("stretch", 2, 16, 0, 0, 16),
    ("stretch", 10, 16, 0, 0, 16),
    ("stretch", 16, 16, 8, 1, 16),
    ("stretch", 30, 8, 0, 0, 16),
    ("stretch", 32, 8, 8, 1, 16),
    ("stretch", 50, 4, 0, 0, 16),
    ("stretch", 64, 4, 8, 1, 16),
    ("stretch", 100, 2, 0, 0, 16),
    ("stretch", 128, 2, 8, 0, 16),
    ("stretch", 200, 1, 0, 0, 16),
    ("stretch", 256, 1, 8, 0, 16),
    ("stretch", 400, 1, 0, 0, 14),
    ("stretch", 700, 1, 0, 0, 8),
    ("de", 4, 8, 0, 0, 16),
    ("de", 40, 4, 0, 0, 16),
    ("de", 80, 2, 0, 0, 16),
    ("de", 150, 1, 0, 0, 16),
    ("de", 240, 1, 0, 0, 15),
    ("de", 256, 1, 8, 0, 13),
    ("de", 300, 1, 0, 0, 12),
    ("snooker", 2, 8, 0, 0, 16),
    ("snooker", 30, 4, 0, 0, 16),
    ("snooker", 60, 2, 0, 0, 16),
    ("snooker", 100, 1, 0, 0, 16),
    ("snooker", 200, 1, 0, 0, 13),
    ("snooker", 256, 1, 8, 0, 10),
    ("snooker", 300, 1, 0, 0, 9),
]
# the register path of stretch with the own row staged like the partner rows
OWN_REG_OFF = [("stretch", 16, 16, 8, 0, 16), ("stretch", 32, 8, 8, 0, 16), ("stretch", 64, 4, 8, 0, 16)]


def _tma_walkers(move, D, R, warps):
    """nwalkers such that, with grid_cap = 1, every warp works through G + 2 tiles of the last split (G = 32 / R
    tiles per batch of draws) and the active counts are not multiples of R (a partial last tile)."""
    P = 4 if move == "snooker" else 2
    G = 32 // R
    m = max((G + 2) * warps * R + 1, -(-2 * D // P) + 1)
    return P * m + 1  # split_starts: the last split gets N // P = m walkers


def _tma_params():
    out = []
    for cell in TMA_CELLS + OWN_REG_OFF:
        for model in ("gauss_iso", "ring", "rosenbrock"):
            own = "" if cell in TMA_CELLS else "-own_reg0"
            for variant in ("capped", "uncapped"):
                out.append(pytest.param(model, cell, variant, id="%s-%s-%d%s-%s" % (cell[0], model, cell[1], own, variant)))
            if cell in TMA_CELLS and cell[1] % 2 == 0:
                out.append(pytest.param(model, cell, "generic", id="%s-%s-%d-tma_rows0" % (cell[0], model, cell[1])))
    return out


@pytest.mark.parametrize("model,cell,variant", _tma_params())
def test_tma_rows_cell(model, cell, variant):
    move, D, R, epl, own, warps = cell
    N = _tma_walkers(move, D, R, warps)
    options = [("tma_own_reg", 0)] if cell in OWN_REG_OFF else []
    if variant == "capped":
        options.append(("grid_cap", 1))
    if variant == "generic":
        options.append(("tma_rows", 0))
    label = "%s %s %d %s" % (move, model, D, variant)
    p = Pair(model, N, D, [(OMOVE[move](), 1.0)], seed=0x7A + D + N, options=options)
    p.free_run(3, label)
    cfg = p.eng.launch_config()
    if variant == "generic":
        _assert_config(cfg, "generic", _lanes_per_walker(D), label=label)
    else:
        _assert_config(cfg, "tma_rows", R, epl, own, warps, label)
        G = 32 // R
        assert cfg["tiles"] == -(-(N // (4 if move == "snooker" else 2)) // R), (label, cfg)
        if variant == "capped":
            assert cfg["grid"] == 1 and cfg["tiles"] // cfg["warps"] >= G + 2, (label, cfg)
    p.single_steps(3, label)


def test_tma_rows_1_sends_long_rows_to_generic():
    """tma_rows = 1 keeps only rows short enough for several walkers per tile on the TMA kernel."""
    for move, D, N in (("stretch", 256, 600), ("de", 150, 400)):
        p = Pair("ring", N, D, [(OMOVE[move](), 1.0)], seed=D, options=[("tma_rows", 1)])
        p.free_run(3, move)
        _assert_config(p.eng.launch_config(), "generic", 32, label=move)
        p.single_steps(2, move)


# ---- generic kernel ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("move", ["stretch", "de", "snooker"])
@pytest.mark.parametrize("D", [3, 17, 33, 65])
def test_generic_odd_ndim(D, move, model):
    """odd ndim goes to the generic kernel at every lanes-per-walker value (4, 8, 16, 32)"""
    N = 4 * D + 37
    label = "%s %s %d" % (move, model, D)
    p = Pair(model, N, D, [(OMOVE[move](), 1.0)], seed=0x6E + D)
    p.free_run(3, label)
    cfg = p.eng.launch_config()
    _assert_config(cfg, "generic", _lanes_per_walker(D), warps=8, label=label)
    assert cfg["threads"] == 256 and cfg["tiles"] == N // (4 if move == "snooker" else 2), cfg
    p.single_steps(3, label)


def test_generic_threads_back_off():
    """snooker on gauss_dense stages 5 rows per walker: above 640-D 8 walkers per CTA exceed 200 KB and the
    launcher halves the block"""
    D = 648
    N = 2 * D
    target, p0 = T.make_config("gauss_dense", N, D, dof=D)  # well conditioned at this size
    p = Pair("gauss_dense", N, D, [(rb.Snooker(), 1.0)], seed=5, target=target, p0=p0)
    p.free_run(3, "snooker 648")
    cfg = p.eng.launch_config()
    _assert_config(cfg, "generic", 32, warps=4, label="snooker 648")
    assert cfg["threads"] == 128, cfg
    p.single_steps(2, "snooker 648")


# ---- gauss_dense off the tensor path ------------------------------------------------------------------------
@pytest.mark.parametrize(
    "move,D",
    [("stretch", 12), ("stretch", 130), ("stretch", 136), ("de", 16), ("de", 64), ("snooker", 16), ("snooker", 64)],
)
def test_gauss_dense_generic(move, D):
    N = 2 * D + 21
    p = Pair("gauss_dense", N, D, [(OMOVE[move](), 1.0)], seed=0xDE + D)
    p.free_run(3, "%s %d" % (move, D))
    _assert_config(p.eng.launch_config(), "generic", _lanes_per_walker(D), label="%s %d" % (move, D))
    p.single_steps(3, "%s %d" % (move, D))


@pytest.mark.parametrize("D", [32, 128])
def test_gauss_dense_nonsymmetric(D):
    """dense_dmma factors the symmetric part of A; the oracle evaluates x^T A x with A as given"""
    N = 4 * D + 13
    target, p0 = T.make_config("gauss_dense", N, D)
    skew = np.triu(np.random.default_rng(D).standard_normal((D, D)), 1) * 0.05
    A = target.icov + skew - skew.T
    tgt = T.GaussDense(A)
    p = Pair("gauss_dense", N, D, [(rb.Stretch(), 1.0)], seed=D, target=tgt, p0=p0)
    p.free_run(3, "nonsym %d" % D)
    _assert_config(p.eng.launch_config(), "dense_dmma", 8, warps=8)
    p.single_steps(3, "nonsym %d" % D)


def test_gauss_dense_indefinite_runs_generic():
    """an A whose Cholesky factorisation fails stays on the generic kernel and still matches"""
    D, N = 32, 77
    target, p0 = T.make_config("gauss_dense", N, D)
    w = np.linalg.eigvalsh(target.icov)
    A = target.icov - 0.5 * (w[0] + w[1]) * np.eye(D)  # one negative eigenvalue
    assert np.linalg.eigvalsh(A)[0] < 0 < np.linalg.eigvalsh(A)[1]
    p = Pair("gauss_dense", N, D, [(rb.Stretch(), 1.0)], seed=3, target=T.GaussDense(A), p0=p0)
    p.free_run(3, "indefinite")
    _assert_config(p.eng.launch_config(), "generic", 8, label="indefinite")
    p.single_steps(3, "indefinite")


# ---- dense_dmma ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("capped", [True, False], ids=["capped", "uncapped"])
@pytest.mark.parametrize("with_mean", [False, True], ids=["mu0", "mu"])
@pytest.mark.parametrize("D", list(range(8, 129, 8)))
def test_dense_dmma_cell(D, with_mean, capped):
    """every width, three splits of 405/404/404 walkers (partial tiles); capped, every consumer warp works
    through at least three tiles: landing-slot reuse and the meta double buffer"""
    N = 1213
    target, p0 = T.make_config("gauss_dense", N, D)
    tgt = T.GaussDense(target.icov, np.linspace(-0.5, 0.5, D) if with_mean else None)
    opts = [("grid_cap", 2)] if capped else []
    label = "dmma %d mean=%s capped=%s" % (D, with_mean, capped)
    p = Pair("gauss_dense", N, D, [(rb.Stretch(nsplits=3), 1.0)], seed=D + 7, options=opts, target=tgt, p0=p0)
    p.free_run(4, label)
    cfg = p.eng.launch_config()
    _assert_config(cfg, "dense_dmma", 8, warps=8, label=label)
    assert cfg["tiles"] == 51, cfg
    if capped:
        assert cfg["grid"] == 2 and cfg["tiles"] // (cfg["grid"] * cfg["warps"]) >= 3, cfg
    coords, lp = p.eng.get_state()
    assert np.array_equal(p.eng.compute_log_prob(coords), lp), label  # same tensor-pipe arithmetic, bit for bit
    p.single_steps(3, label)


def test_dense_dmma_options_change_nothing():
    """dmma_group (cooperative launch with the in-kernel grid barrier), pdl, dmma_stagger and grid_cap only
    change how the work is launched: every combination gives the same bits"""
    N, D, nsteps = 1213, 64, 4
    target, p0 = T.make_config("gauss_dense", N, D)
    tgt = T.GaussDense(target.icov, np.linspace(-0.5, 0.5, D))
    ref = None
    for group in (1, 2, 7):
        for pdl in (0, 1):
            for stagger in (0, 1):
                for cap in (0, 3):
                    opts = [("dmma_group", group), ("pdl", pdl), ("dmma_stagger", stagger), ("grid_cap", cap)]
                    p = Pair("gauss_dense", N, D, [(rb.Stretch(nsplits=3), 1.0)], seed=11, options=opts, target=tgt, p0=p0)
                    acc = p.eng.step(p.sched, nsteps)
                    coords, lp = p.eng.get_state()
                    got = (acc, coords, lp, p.eng.naccepted())
                    assert p.eng.last_kernel_name() == "dense_dmma"
                    if ref is None:
                        acc_o = p.o.run(nsteps)
                        assert np.array_equal(acc, acc_o) and np.array_equal(coords, p.o.coords)
                        np.testing.assert_allclose(lp, p.o.log_prob, rtol=1e-11, atol=1e-11)
                        ref = got
                    for a, b in zip(got, ref):
                        assert np.array_equal(a, b), opts


# ---- one input through every path ---------------------------------------------------------------------------
CROSS = [
    # model, move, ndim, nwalkers, option sets (the first is the reference)
    ("gauss_iso", "stretch", 32, 2301, [dict(tma_rows=r, tma_own_reg=o) for r in (2, 1, 0) for o in (1, 0)]),
    ("ring", "stretch", 256, 1201, [dict(tma_rows=r) for r in (2, 1, 0)]),
    ("rosenbrock", "de", 128, 1001, [dict(tma_rows=r) for r in (2, 1, 0)]),
    ("gauss_iso", "snooker", 60, 2401, [dict(tma_rows=r) for r in (2, 1, 0)]),
    ("gauss_dense", "stretch", 64, 1201, [dict(dense_dmma=d) for d in (1, 0)]),
]


@pytest.mark.parametrize("model,move,D,N,paths", CROSS, ids=["%s-%s-%d" % c[:3] for c in CROSS])
def test_cross_path_equality(model, move, D, N, paths):
    """the same state and seed through every kernel that can take it, each with several grid caps: accept
    masks identical, stretch / DE coordinates bit-identical (every path rounds the same sub / mul / add
    sequence), snooker coordinates and log-probabilities to 1e-12 (summation order); within one path the
    grid cap changes nothing at all"""
    target, p0 = T.make_config(model, N, D)
    ref = None
    for path in paths:
        path_ref = None
        for cap in (0, 1, 5):
            opts = list(path.items()) + [("grid_cap", cap)]
            p = Pair(model, N, D, [(OMOVE[move](), 1.0)], seed=99, options=opts, target=target, p0=p0)
            if ref is None:
                lp0 = p.lp0
                p.free_run(3, "reference path %s" % opts)
                p.eng.set_state(p0, lp0)
                p.eng.set_rng(99, 0)
            else:
                p.eng.set_state(p0, lp0)  # one input: the reference path's initial log-probabilities
            got = (p.eng.step(p.sched, 3),) + p.eng.get_state()
            label = "%s %s" % (opts, p.eng.launch_config())
            if ref is None:
                ref = got
            if path_ref is None:
                path_ref = got
            for a, b in zip(got, path_ref):
                assert np.array_equal(a, b), label
            assert np.array_equal(got[0], ref[0]), label
            if move == "snooker":
                np.testing.assert_allclose(got[1], ref[1], rtol=1e-12, atol=1e-12, err_msg=label)
            else:
                assert np.array_equal(got[1], ref[1]), label
            rtol = 1e-11 if model == "gauss_dense" else 1e-12  # see _lp_tols
            np.testing.assert_allclose(got[2], ref[2], rtol=rtol, atol=rtol, err_msg=label)


# ---- non-finite guards on every variant ---------------------------------------------------------------------
GUARDS = [
    # model, move, ndim, nwalkers, options, (kernel, width, epl, own_reg)
    ("gauss_iso", "stretch", 32, 301, {}, ("tma_rows", 8, 8, 1)),
    ("gauss_iso", "stretch", 32, 301, {"tma_own_reg": 0}, ("tma_rows", 8, 8, 0)),
    ("ring", "de", 256, 601, {}, ("tma_rows", 1, 8, 0)),
    ("ring", "stretch", 30, 301, {}, ("tma_rows", 8, 0, 0)),
    ("rosenbrock", "de", 40, 301, {}, ("tma_rows", 4, 0, 0)),
    ("gauss_iso", "stretch", 200, 601, {}, ("tma_rows", 1, 0, 0)),
    ("gauss_iso", "stretch", 33, 301, {}, ("generic", 16, 0, 0)),
    ("ring", "de", 33, 301, {}, ("generic", 16, 0, 0)),
    ("gauss_dense", "stretch", 32, 301, {}, ("dense_dmma", 8, 0, 0)),
]


@pytest.mark.parametrize("model,move,D,N,opts,variant", GUARDS, ids=["%s-%s-%d-%s" % (g[0], g[1], g[2], "-".join(map(str, g[5]))) for g in GUARDS])
def test_nonfinite_proposal_raises(model, move, D, N, opts, variant):
    """the last element of every row at +-1.5e308, alternating across walkers: a proposal between two walkers of
    opposite sign overflows, and the step raises like compute_log_prob (ensemble.py:476-477)"""
    p = Pair(model, N, D, [(OMOVE[move](), 1.0)], seed=D, options=list(opts.items()))
    p.free_run(1, "finite")
    _assert_config(p.eng.launch_config(), *variant)
    bad = p.p0.copy()
    bad[:, -1] = 1.5e308 * (-1.0) ** np.arange(N)
    p.eng.set_state(bad, np.zeros(N))
    with pytest.raises(ValueError, match="infinite"):
        p.eng.step(p.sched, 1)
    # the engine steps normally from a finite state afterwards
    p.single_steps(2, "after the error")


# ---- tiny ensembles ----------------------------------------------------------------------------------------
TINY = [
    # model, move, ndim, nwalkers, nsplits, live_dangerously, kernel
    ("gauss_iso", "stretch", 32, 64, 2, False, "tma_rows"),
    ("rosenbrock", "stretch", 17, 34, 2, False, "generic"),
    ("gauss_dense", "stretch", 16, 32, 2, False, "dense_dmma"),
    ("gauss_iso", "stretch", 32, 40, 2, True, "tma_rows"),
    ("ring", "de", 40, 50, 2, True, "tma_rows"),
    ("gauss_dense", "stretch", 24, 30, 2, True, "dense_dmma"),
    # five sets of 4 walkers: fewer than one tile (R = 16, 8, 8)
    ("gauss_iso", "stretch", 10, 20, 5, False, "tma_rows"),
    ("ring", "de", 4, 20, 5, False, "tma_rows"),
    ("gauss_dense", "stretch", 16, 36, 5, False, "dense_dmma"),
]


@pytest.mark.parametrize("model,move,D,N,nsplits,live,kernel", TINY, ids=["%s-%s-%dx%d-p%d" % (t[0], t[1], t[3], t[2], t[4]) for t in TINY])
def test_tiny_ensemble(model, move, D, N, nsplits, live, kernel):
    omove = OMOVE[move](nsplits=nsplits, live_dangerously=live)
    dmove = {"stretch": dmoves.StretchMove, "de": dmoves.DEMove}[move](nsplits=nsplits, live_dangerously=live)
    p = Pair(model, N, D, [(omove, 1.0)], seed=N + D, dmoves_=[(dmove, 1.0)])
    p.free_run(4, "tiny")
    assert p.eng.launch_config()["kernel"] == kernel
    p.single_steps(3, "tiny")
