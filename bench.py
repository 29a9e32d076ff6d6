#!/usr/bin/env python
"""Headline benchmark: walker-steps/s of the red-blue walker update.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one full ensemble step (every walker proposed once = the P
half-steps of ``RedBlueMove.propose``).  Headline workload = BASELINE.json's
metric configuration: 65 536 walkers, 128-D correlated Gaussian (dense inverse
covariance), StretchMove(a=2), randomised split, fp64.  With N GPUs the SAME
65 536 walkers are sharded by row block over the N ranks (strong scaling, config
3 of BASELINE.json -- what north_star's ">= 6x at 8 GPUs" is quoted on); the
weak-scaling run (65 536 walkers PER GPU) is reported beside it in ``"weak"``.

Prints ONE JSON line (rank 0).  ``value`` is device-timed (CUDA events on the
engine's stream, max over ranks) with the state resident in HBM and L2 flushed
before every step; ``e2e`` is the same metric through the public API
``EnsembleSampler.run_mcmc`` with pinned HOST buffers, copies inside the timed
region (sharded: every rank moves only the rows it owns).  ``configs`` holds
short runs of BASELINE.json's other configurations.  ``--impl reference`` times
the UNMODIFIED reference package (``oracle/_ref``: ``vectorize=True`` and
``multiprocessing.Pool``) on the host cores, with the numpy oracle port beside it,
each over exactly ``--steps`` steps after ``--warmup``.
"""

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "walker-steps/sec (nwalkers x iters / s)"
MODEL_SEED, INIT_SEED, SAMPLER_SEED = 20240, 20241, 0x656D636565B200
REF_ZIP = os.path.join(ROOT, "oracle", "_ref", "emcee_reference.zip")
FP64_PEAK_RECORDED = 37.0  # TFLOP/s, eb_microbench DMMA m8n8k4 (profiles/r01_fp64_microbench.txt)
DUMP_BYTES, DUMP_SEED = 64 * 10**6, 0xD0  # --dump-outputs: size cap of all files together, walker-sample seed


# --------------------------------------------------------------------------
# synthetic workloads (SURVEY 8d / DESIGN.md); plain numpy parameter generation
# --------------------------------------------------------------------------
def make_workload(name, nwalkers, ndim):
    rng_m = np.random.default_rng(MODEL_SEED)
    rng_p = np.random.default_rng(INIT_SEED)
    w = {"name": name, "nwalkers": nwalkers, "ndim": ndim}
    if name == "gauss_dense":
        v = rng_m.standard_normal((ndim + 1, ndim))  # random_cov(ndim, dof=1), document/plots/oned.py:21-25
        cov = (v.T @ v) / (ndim + 1)
        icov = np.linalg.inv(cov)
        w["icov"] = 0.5 * (icov + icov.T)
        w["p0"] = rng_p.standard_normal((nwalkers, ndim))
        w["moves"] = "stretch"
    elif name == "gauss_iso":
        w["p0"] = rng_p.standard_normal((nwalkers, ndim))
        w["moves"] = "stretch"
    elif name == "ring":
        w["radius"], w["sigma"] = 5.0, 0.5
        w["p0"] = rng_p.standard_normal((nwalkers, ndim)) * (5.0 / np.sqrt(ndim))
        w["moves"] = "stretch"
    elif name == "rosenbrock":
        w["p0"] = 1.0 + 0.1 * rng_p.standard_normal((nwalkers, ndim))
        w["moves"] = "de+snooker"
    else:
        raise ValueError(name)
    return w


def flops_bytes_per_walker_step(w):
    """Algorithmic work of one walker-step (SURVEY 8d, BASELINE.md section 4): fp64 bytes with the
    row write counted unconditionally, and flops of proposal + log-prob.  For the dense Gaussian TWO
    flop conventions exist and both are returned: ``executed`` = D(D+1) + 2D for the factored form
    -0.5 |L^T x|^2 the kernel evaluates (A = L L^T), and ``contract`` = 2D^2 + 3D for the unfactored
    x^T A x that SURVEY 8d quotes.  The roofline fraction reported as ``frac`` uses ``executed`` (the
    conservative one); ``frac_contract`` uses the other."""
    D = w["ndim"]
    if w["moves"] == "stretch":
        nbytes, prop = 24 * D + 24, 3 * D
    else:  # 0.8 DE + 0.2 snooker
        nbytes = 0.8 * (32 * D + 24) + 0.2 * (40 * D + 24)
        prop = 0.8 * 3 * D + 0.2 * 10 * D
    lp = {"gauss_dense": D * (D + 1) + 2 * D, "gauss_iso": 2 * D, "ring": 2 * D + 6, "rosenbrock": 9 * (D - 1)}[w["name"]]
    lp_contract = 2 * D * D + 3 * D if w["name"] == "gauss_dense" else lp
    return prop + lp, prop + lp_contract, nbytes


# --------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region
    (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL,
            )
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)), reasons=sorted(reasons), samples=len(sm))
        return out


def dump_outputs(dirname, coords, log_prob, naccepted):
    """``--dump-outputs``: the ensemble state the timed steps left -- what ``run_mcmc`` hands its caller --
    and the per-walker acceptance counts, as ``<dirname>/{coords,log_prob,naccepted}.npy`` (float64).  When
    they would exceed DUMP_BYTES together, the same fixed seeded sample of walkers is taken from each and
    its row numbers are written as ``walkers.npy``."""
    out = {"coords": coords, "log_prob": log_prob, "naccepted": naccepted.astype(np.float64)}
    n, d = coords.shape
    per_walker = 8 * (d + 2)
    if n * per_walker > DUMP_BYTES:
        k = (DUMP_BYTES - 4096) // (per_walker + 8)  # 4096: room for the .npy headers
        rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False))
        out = {name: a[rows] for name, a in out.items()}
        out["walkers"] = rows.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def kernel_traffic(kernel):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/traffic.json, written by scripts/summarize_ncu.py), or None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return t.get(kernel)
    except Exception:
        return None


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def blas_threads():
    try:
        from threadpoolctl import threadpool_info

        n = [p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"]
        return int(max(n)) if n else 1
    except Exception:
        return 1


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# --------------------------------------------------------------------------
# CPU arms (bench.py may execute oracle/ and oracle/_ref only here)
# --------------------------------------------------------------------------
def oracle_sampler(w, seed):
    from oracle import redblue as rb
    from oracle import targets as T

    D = w["ndim"]
    target = {
        "gauss_dense": lambda: T.GaussDense(w["icov"]),
        "gauss_iso": lambda: T.GaussIso(D),
        "ring": lambda: T.Ring(D, w["radius"], w["sigma"]),
        "rosenbrock": lambda: T.Rosenbrock(D),
    }[w["name"]]()
    moves = [(rb.Stretch(), 1.0)] if w["moves"] == "stretch" else [(rb.DE(), 0.8), (rb.Snooker(), 0.2)]
    o = rb.OracleSampler(w["nwalkers"], D, target, moves, seed=seed)
    o.set_state(w["p0"])
    return o


def time_oracle(w, steps, warmup):
    o = oracle_sampler(w, SAMPLER_SEED)
    o.run(warmup)
    t0 = time.perf_counter()
    o.run(steps)
    dt = time.perf_counter() - t0
    return w["nwalkers"] * steps / dt, dt


# the log-probabilities handed to the UNMODIFIED reference: module-level so that
# multiprocessing.Pool can pickle them by name (docs/tutorials/parallel.ipynb:183-192)
_REF = {}


def _ref_logp_vec(x):
    k = _REF["name"]
    if k == "gauss_dense":
        return -0.5 * np.sum((x @ _REF["icov"]) * x, axis=-1)
    if k == "gauss_iso":
        return -0.5 * np.sum(x * x, axis=-1)
    if k == "ring":
        d = np.sqrt(np.sum(x * x, axis=-1)) - _REF["radius"]
        return -(d * d) / (2.0 * _REF["sigma"] ** 2)
    x0, x1 = x[..., :-1], x[..., 1:]
    return -np.sum(100.0 * (x1 - x0 * x0) ** 2 + (1.0 - x0) ** 2, axis=-1)


def _ref_logp_row(x):
    return float(_ref_logp_vec(x))


def import_reference():
    """The unmodified reference package from oracle/_ref (see oracle/make_ref.py), or None."""
    if not os.path.exists(REF_ZIP):
        return None
    if REF_ZIP not in sys.path:
        sys.path.insert(0, REF_ZIP)
    import emcee

    assert REF_ZIP in emcee.__file__, emcee.__file__
    return emcee


def time_reference(w, steps, warmup, pool_steps, repeats=3):
    """walker-steps/s of the unmodified reference on this host: (i) ``vectorize=True`` with a numpy
    batched log-prob, (ii) ``multiprocessing.Pool(ncores)`` with a per-walker log-prob and BLAS pinned
    to one thread (docs/tutorials/parallel.ipynb:40,52,183-192).  Median of ``repeats``."""
    emcee = import_reference()
    if emcee is None:
        return None
    _REF.clear()
    _REF.update({k: w[k] for k in ("name", "icov", "radius", "sigma") if k in w})
    N, D = w["nwalkers"], w["ndim"]
    mv = (emcee.moves.StretchMove() if w["moves"] == "stretch"
          else [(emcee.moves.DEMove(), 0.8), (emcee.moves.DESnookerMove(), 0.2)])
    kw = dict(store=False, skip_initial_state_check=True)
    np.random.seed(1234)
    out = {}
    s = emcee.EnsembleSampler(N, D, _ref_logp_vec, moves=mv, vectorize=True)
    s.run_mcmc(w["p0"], max(1, warmup), **kw)
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        s.run_mcmc(None, steps, **kw)
        ts.append(time.perf_counter() - t0)
    out["vectorize"] = {"value": N * steps / float(np.median(ts)), "steps": steps, "seconds": float(np.median(ts))}
    if pool_steps > 0:
        import multiprocessing as mp

        import contextlib

        try:
            from threadpoolctl import threadpool_limits

            one_blas_thread = threadpool_limits(limits=1)
        except Exception:
            one_blas_thread = contextlib.nullcontext()
        ncores = host_cores()
        with one_blas_thread, mp.get_context("fork").Pool(ncores) as pool:
            s = emcee.EnsembleSampler(N, D, _ref_logp_row, moves=mv, pool=pool)
            s.run_mcmc(w["p0"], max(1, warmup), **kw)
            ts = []
            for _ in range(repeats):
                t0 = time.perf_counter()
                s.run_mcmc(None, pool_steps, **kw)
                ts.append(time.perf_counter() - t0)
        out["pool"] = {"value": N * pool_steps / float(np.median(ts)), "steps": pool_steps,
                       "seconds": float(np.median(ts)), "processes": ncores}
    return out


def cpu_arms(w, steps, warmup, pool_steps, keep_going=True):
    """The CPU baseline object: the unmodified reference (best of its two own execution modes) when
    oracle/_ref holds it, with the oracle port beside it; else the port alone, named as such.  A failing
    reference is reported in the object when `keep_going` (the GPU arm's line), else raised."""
    port_v, port_dt = time_oracle(w, steps, warmup)
    ref = None
    try:
        ref = time_reference(w, steps, warmup, pool_steps)
    except Exception as e:
        if not keep_going:
            raise
        ref = {"error": repr(e)}  # never lose the GPU headline over the baseline beside it
    what = "%dx%d %s" % (w["nwalkers"], w["ndim"], w["name"])
    if ref and "vectorize" in ref:
        best_mode = max((k for k in ("vectorize", "pool") if k in ref), key=lambda k: ref[k]["value"])
        return {
            "value": ref[best_mode]["value"], "unit": "walker-steps/s", "cores": host_cores(), "kind": "reference",
            "sample": "unmodified dfm/emcee@8ab6c0f (oracle/_ref), %s: vectorize=True %d steps x3 (median %.2f s, BLAS threads=%d)%s; "
                      "best mode = %s; numpy oracle port beside it" % (
                          what, ref["vectorize"]["steps"], ref["vectorize"]["seconds"], blas_threads(),
                          "; Pool(%d) per-walker log-prob, BLAS threads=1, %d steps x3 (median %.2f s)" % (
                              ref["pool"]["processes"], ref["pool"]["steps"], ref["pool"]["seconds"]) if "pool" in ref else "",
                          best_mode),
            "reference_vectorize": ref["vectorize"]["value"],
            "reference_pool": ref.get("pool", {}).get("value"),
            "port": port_v, "blas_threads": blas_threads(), "numpy": np.__version__,
        }
    return {"value": port_v, "unit": "walker-steps/s", "cores": blas_threads(), "kind": "port",
            "sample": "%d steps of %s on the numpy oracle port (%.1f s; BLAS threads=%d, rest single-threaded); "
                      "unmodified reference not timed: %s" % (
                          steps, what, port_dt, blas_threads(),
                          (ref or {}).get("error", "oracle/_ref/emcee_reference.zip absent (oracle/make_ref.py found no "
                                                   "readable reference checkout)")),
            "port": port_v}


def run_reference(args, dist):
    """``--impl reference``: the reference's own CPU implementation of the path on this box's host
    cores, every arm timed over exactly ``--steps`` steps after ``--warmup`` (the Pool arm too, unless
    ``--cpu-pool-steps 0`` skips it).  Rank 0 only."""
    if dist.rank != 0:
        return
    w = make_workload(args.workload, args.nwalkers, args.ndim)
    steps = args.steps
    t0 = time.perf_counter()
    cpu = cpu_arms(w, steps, args.warmup, steps if args.cpu_pool_steps > 0 else 0, keep_going=False)
    value = cpu["value"]
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": "walker-steps/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * w["nwalkers"] / value,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(args, w, 1, w["nwalkers"], "strong"),
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": "walker-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line))


def workload_config(args, w, world, n_total, scaling):
    mv = "StretchMove(a=2)" if w["moves"] == "stretch" else "0.8 DEMove + 0.2 DESnookerMove"
    if world > 1:
        where = "%d walkers sharded by row block over %d GPUs (%d per GPU, %s scaling)" % (
            n_total, world, n_total // world, scaling)
    else:
        where = "1 GPU"
    return {
        "workload": "%s %dx%d, %s, fp64, randomize_split=True, %s" % (w["name"], n_total, w["ndim"], mv, where),
        "nwalkers_total": n_total,
        "ndim": w["ndim"],
        "l2": args.l2_note,
        "comm": args.comm if world > 1 else "none",
    }


# --------------------------------------------------------------------------
# the B200 arm
# --------------------------------------------------------------------------
def device_model(w):
    from emcee_b200 import models

    return {
        "gauss_dense": lambda: models.GaussianDense(w["icov"]),
        "gauss_iso": lambda: models.GaussianIso(),
        "ring": lambda: models.Ring(w["radius"], w["sigma"]),
        "rosenbrock": lambda: models.Rosenbrock(),
    }[w["name"]]()


def device_moves(w):
    from emcee_b200 import moves

    return moves.StretchMove() if w["moves"] == "stretch" else [(moves.DEMove(), 0.8), (moves.DESnookerMove(), 0.2)]


def build_sampler(args, w, dist, gather_results=True, pinned=False):
    import emcee_b200

    s = emcee_b200.EnsembleSampler(w["nwalkers"], w["ndim"], device_model(w), moves=device_moves(w), seed=SAMPLER_SEED,
                                   device=dist.local_rank, pinned_results=pinned)
    if dist.world > 1:
        s.attach(dist, args.comm, gather_results=gather_results)
    eng = s._engine
    if args.dmma_group > 0:
        eng.set_option("dmma_group", args.dmma_group)
    if args.no_tma_rows:
        eng.set_option("tma_rows", 0)
    if args.tma_rows:
        eng.set_option("tma_rows", args.tma_rows)
    if args.no_stagger:
        eng.set_option("dmma_stagger", 0)
    if args.no_pdl:
        eng.set_option("pdl", 0)
    if args.no_own_reg:
        eng.set_option("tma_own_reg", 0)
    return s


def measure_device(args, w, dist, steps, warmup, flush, clocks=None, dump_dir=None):
    """Device-resident throughput: CUDA events on the engine's stream around exactly `steps` steps
    (per-step brackets with an L2 flush before each when `flush`), max over ranks.  With `dump_dir`, the
    state after those steps is written there (rank 0)."""
    s = build_sampler(args, w, dist)
    eng = s._engine
    eng.set_option("l2_flush", 1 if flush else 0)
    sched = s._schedule()
    eng.set_state(w["p0"])
    eng.step(sched, warmup, want_accepted=False)
    dist.barrier()
    if clocks is not None:
        clocks.start()
    t0 = time.perf_counter()
    eng.step(sched, steps, want_accepted=False)  # synchronous at return
    wall = time.perf_counter() - t0
    dist.barrier()
    ck = clocks.stop() if clocks is not None else None
    ms, launches = eng.last_step_timing()
    ms, wall = dist.max(ms), dist.max(wall)
    if dump_dir is not None:
        # read before the clock probe below steps the ensemble further; collective on a sharded engine
        coords, log_prob = eng.get_state()
        naccepted = eng.naccepted()
        if dist.rank == 0:
            dump_outputs(dump_dir, coords, log_prob, naccepted)
    out = {"ms": ms, "wall": wall, "launches": launches, "kernel": eng.last_kernel_name(),
           "value": w["nwalkers"] * steps / (ms * 1e-3)}
    if ck is not None:
        ck["source"] = "timed region"
        if ck["samples"] < 3:
            # the timed region is shorter than nvidia-smi can resolve: repeat the same workload for ~0.7 s
            # more (the repeat count comes from the max-over-ranks time, so every rank runs the same
            # number of steps: they contain cross-rank barriers)
            reps = max(1, min(200, int(0.7 / max(ms * 1e-3, 1e-4))))
            probe = ClockSampler(dist.local_rank)
            probe.start()
            for _ in range(reps):
                eng.step(sched, steps, want_accepted=False)
            ck2 = probe.stop()
            if ck2["samples"] > ck["samples"]:
                ck = ck2
                ck["source"] = "same workload repeated for ~0.7 s right after the timed region (region too short to sample)"
        out["clocks"] = ck
    eng.close()
    dist.barrier()
    return out


def measure_e2e(args, w, dist, steps, warmup):
    """The call a user makes: run_mcmc(p0, K, store=False) with pinned host buffers -- H2D of the
    initial state, K steps, D2H of the final state (sharded: each rank moves the rows it owns)."""
    from emcee_b200 import _lib

    N, D = w["nwalkers"], w["ndim"]
    s = build_sampler(args, w, dist, gather_results=False, pinned=True)
    p0 = _lib.pinned_empty((N, D))
    p0[...] = w["p0"]
    kw = dict(store=False, skip_initial_state_check=True)
    s.run_mcmc(p0, max(3, warmup // 4), **kw)
    dist.barrier()
    t0 = time.perf_counter()
    last = s.run_mcmc(p0, steps, **kw)
    wall = dist.max(time.perf_counter() - t0)
    rows = s.owned_rows
    assert np.all(np.isfinite(last.log_prob[rows]))
    s._engine.close()
    dist.barrier()
    return {"value": N * steps / wall, "unit": "walker-steps/s",
            "h2d_bytes_per_step": N * D * 8 / steps, "d2h_bytes_per_step": (N * D * 8 + N * 8) / steps,
            "call": "EnsembleSampler.run_mcmc(p0_pinned_host, %d, store=False): H2D initial state + %d steps + D2H final state, "
                    "wall clock%s" % (steps, steps, "; bytes summed over ranks, each rank moves only its own row block" if dist.world > 1 else "")}


def parity_check(args, w, dist, steps=5):
    """Multi-GPU correctness inside the bench: the sharded run's global state after `steps` steps must
    be identical on every rank AND bit-identical to a 1-rank run of the same ensemble."""
    import emcee_b200

    kw = dict(store=False, skip_initial_state_check=True)
    s = build_sampler(args, w, dist, gather_results=True)
    last = s.run_mcmc(w["p0"], steps, **kw)
    nacc = s._engine.naccepted()
    digest = hashlib.sha256(last.coords.tobytes() + last.log_prob.tobytes() + nacc.tobytes()).hexdigest()
    s._engine.close()
    digests = dist.allgather(digest)
    ok = all(d == digests[0] for d in digests)
    if dist.rank == 0:
        one = emcee_b200.EnsembleSampler(w["nwalkers"], w["ndim"], device_model(w), moves=device_moves(w), seed=SAMPLER_SEED,
                                         device=dist.local_rank)
        ref = one.run_mcmc(w["p0"], steps, **kw)
        ok = ok and np.array_equal(ref.coords, last.coords) and np.array_equal(ref.log_prob, last.log_prob) \
            and np.array_equal(one._engine.naccepted(), nacc)
        one._engine.close()
    ok = bool(dist.bcast(ok))
    if not ok:
        raise SystemExit("bench.py: multi-GPU parity check FAILED (%s, %d ranks): sharded run differs from the 1-rank run"
                         % (w["name"], dist.world))
    return True


def rooflines(args, w, value_per_gpu, fp64_peak, fp64_src):
    flops, flops_contract, nbytes = flops_bytes_per_walker_step(w)
    peaks = measured_peaks()
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "B200_PROFILING.md fallback 6650 GB/s (of fallback)"
    ach_gbs = value_per_gpu * nbytes / 1e9
    ach_tf = value_per_gpu * flops / 1e12
    hbm = {"bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak,
           "traffic": None, "peak_source": hbm_src,
           "note": "algorithmic bytes/walker-step = %g (SURVEY 8d) over the whole timed region (launch gaps included)" % nbytes}
    if w["name"] == "gauss_dense" and fp64_peak:
        main = {"bound": "tensor", "achieved": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach_tf / fp64_peak,
                "frac_contract": value_per_gpu * flops_contract / 1e12 / fp64_peak,
                "traffic": kernel_traffic("dense_dmma"), "peak_source": fp64_src,
                "flops_per_walker_step": {"executed": flops, "contract": flops_contract},
                "note": "frac counts the EXECUTED flops/walker-step = %g (triangular D(D+1)+2D log-prob + 3D proposal, "
                        "BASELINE.md section 4); frac_contract counts SURVEY 8d's unfactored 2D^2+3D = %g; whole timed region"
                        % (flops, flops_contract)}
        return main, hbm
    return hbm, hbm


# BASELINE.json's other configurations: short runs, L2-warm (the state of a real run), reported per config
def other_configs(args, dist):
    world = dist.world
    specs = [
        ("config4 rosenbrock 16384x256 0.8 DE + 0.2 snooker", "rosenbrock", 16384, 256),
        ("config5 ring %dx32 stretch%s" % (262144 if world == 1 else 32768 * world,
                                           "" if world == 1 else " (weak: 32768 per GPU)"),
         "ring", 262144 if world == 1 else 32768 * world, 32),
    ]
    if world == 1:  # the single-GPU configurations of BASELINE.json
        specs = [
            ("config1 gauss_iso 32x5 stretch (quickstart shape)", "gauss_iso", 32, 5),
            ("config2 gauss_dense 4096x128 stretch", "gauss_dense", 4096, 128),
        ] + specs
    out = {}
    for label, name, n, d in specs:
        try:
            w = make_workload(name, n, d)
            steps = 200 if n * d <= (1 << 22) else 60
            m = measure_device(args, w, dist, steps, 10, False)
            roof, _ = rooflines(args, w, m["value"] / world, FP64_PEAK_RECORDED, "recorded eb_microbench DMMA peak")
            out[label] = {"value": m["value"], "ms_per_step": m["ms"] / steps, "steps": steps, "kernel": m["kernel"],
                          "n_gpus": world, "l2": "warm", "roofline": {k: roof[k] for k in ("bound", "achieved", "peak", "unit", "frac")}}
        except BaseException as e:  # a side run must never take the headline down
            if isinstance(e, KeyboardInterrupt):
                raise
            out[label] = {"error": repr(e)}
    return out


def run_b200(args, dist):
    from emcee_b200 import _lib

    world = dist.world
    D = args.ndim
    n_strong = args.nwalkers
    if n_strong % world:
        raise SystemExit("--nwalkers must be divisible by the number of GPUs")
    w = make_workload(args.workload, n_strong, D)

    # ---- headline: the metric configuration, sharded over the ranks (strong scaling) -------------
    parity = parity_check(args, w, dist) if world > 1 else None
    head = measure_device(args, w, dist, args.steps, args.warmup, args.l2_flush, ClockSampler(dist.local_rank),
                          dump_dir=args.dump_outputs)
    e2e = measure_e2e(args, w, dist, args.steps, args.warmup)

    # ---- weak scaling beside it: the same walkers PER GPU ----------------------------------------
    weak = None
    if world > 1:
        ww = make_workload(args.workload, n_strong * world, D)
        weak_parity = parity_check(args, ww, dist)
        wm = measure_device(args, ww, dist, args.steps, args.warmup, args.l2_flush)
        we = measure_e2e(args, ww, dist, args.steps, args.warmup)
        weak = {"value": wm["value"], "unit": "walker-steps/s", "ms_per_step": wm["ms"] / args.steps,
                "nwalkers_total": n_strong * world, "nwalkers_per_gpu": n_strong, "e2e": we, "gpu_launches": wm["launches"],
                "parity_checked": weak_parity, "kernel": wm["kernel"]}

    configs = None if args.no_configs else other_configs(args, dist)

    if dist.rank != 0:
        return

    fp64_peak, fp64_src = None, ("fp64 issue-rate peak measured on this GPU by eb_microbench (max of DMMA m8n8k4 and DFMA); "
                                 "MEASURED_PEAKS.json has no fp64 entry")
    if args.no_microbench:
        fp64_peak, fp64_src = FP64_PEAK_RECORDED, "recorded eb_microbench DMMA m8n8k4 peak (profiles/r01_fp64_microbench.txt)"
    else:
        try:
            fp64_peak = max(_lib.microbench(1, 16), _lib.microbench(0, 32))
        except Exception:
            fp64_peak, fp64_src = FP64_PEAK_RECORDED, "recorded eb_microbench DMMA m8n8k4 peak (microbench failed)"
    roofline, roofline_hbm = rooflines(args, w, head["value"] / world, fp64_peak, fp64_src)
    if weak is not None:
        wr, _ = rooflines(args, w, weak["value"] / world, fp64_peak, fp64_src)
        weak["roofline_frac"] = wr["frac"]

    # ---- CPU baseline beside it (bounded sample, rank 0 only, N=1 only) ------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_arms(w, args.cpu_steps, 2, args.cpu_pool_steps)

    ck = head["clocks"]
    line = {
        "metric": METRIC, "value": head["value"], "unit": "walker-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": head["ms"] / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, w, world, n_strong, "strong"),
        "clocks": {"sm_mhz": ck["sm_mhz"], "sm_max_mhz": ck["sm_max_mhz"], "reasons": ck["reasons"], "samples": ck["samples"],
                   "source": ck["source"]},
        "e2e": e2e,
        "gpu_launches": head["launches"],
        "kernel": head["kernel"],
        "wall_ms_per_step": 1e3 * head["wall"] / args.steps,
        "roofline": roofline,
        "roofline_hbm": roofline_hbm,
        "cpu_baseline": cpu,
    }
    if world > 1:
        line["parity_checked"] = parity
        line["weak"] = weak
    if configs is not None:
        line["configs"] = configs
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="gauss_dense", choices=["gauss_dense", "gauss_iso", "ring", "rosenbrock"])
    ap.add_argument("--nwalkers", type=int, default=65536, help="walkers of the metric configuration (in total: strong scaling)")
    ap.add_argument("--ndim", type=int, default=128)
    ap.add_argument("--comm", default="p2p", choices=["allgather", "p2p"],
                    help="multi-GPU exchange: NVLink peer-memory pull (default) or one ncclAllGather per split")
    ap.add_argument("--no-l2-flush", dest="l2_flush", action="store_false")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the short runs of BASELINE.json's other configurations")
    ap.add_argument("--no-microbench", action="store_true",
                    help="do not launch the fp64 peak micro-benchmarks (for ncu launch lists); use the recorded peak")
    ap.add_argument("--tma-rows", type=int, default=0, help="tma_rows option value (1: short rows only, 2: long rows too)")
    ap.add_argument("--no-tma-rows", action="store_true", help="HBM-bound models: use the generic kernel instead of tma_rows")
    ap.add_argument("--no-own-reg", action="store_true", help="tma_rows: stage the own rows through the TMA unit as well")
    ap.add_argument("--no-stagger", action="store_true", help="dense_dmma: all pairs request their first tile at once")
    ap.add_argument("--no-pdl", action="store_true", help="dense_dmma: plain stream-ordered launches instead of programmatic dependent launches")
    ap.add_argument("--dmma-group", type=int, default=0, help="half-steps per persistent dense_dmma launch (0: library default)")
    ap.add_argument("--cpu-steps", type=int, default=20, help="steps of the cpu_baseline object beside the GPU arm")
    ap.add_argument("--cpu-pool-steps", type=int, default=2,
                    help="steps of the reference's Pool arm in that object (0: skip it; with --impl reference the "
                         "Pool arm times --steps steps, and 0 skips it)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the state the timed steps of the headline run left as DIR/<name>.npy, so that two "
                         "builds can be compared output for output (the inputs are seeded)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes what the timed GPU path computed; it needs --impl b200")
    args.warmup = max(3, args.warmup)
    args.l2_note = (
        "L2 flushed between timed steps (256 MiB device memset, outside the per-step CUDA-event brackets)"
        if args.l2_flush else
        "no flush: the ensemble (N*D*8 B) stays L2-resident across steps, as it does in a real run"
    )
    from emcee_b200.dist import Rendezvous

    dist = Rendezvous()
    if dist.world != args.gpus and dist.world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, dist.world))
    try:
        if args.impl == "reference":
            run_reference(args, dist)
        else:
            run_b200(args, dist)
    finally:
        dist.close()


if __name__ == "__main__":
    main()
