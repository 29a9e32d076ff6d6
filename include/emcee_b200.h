/*
 * emcee_b200.h -- C ABI of the B200-native ensemble-MCMC walker-update engine.
 *
 * This is the drop-in boundary for the hot path of dfm/emcee (reference @ 8ab6c0f,
 * pure Python, no FFI of its own).  Each entry point below names the reference
 * interface it replaces (file:line relative to the reference root).  The Python
 * host side (emcee_b200/ensemble.py, moves/, state.py) binds these with ctypes
 * and mirrors EnsembleSampler / moves.Move / State; INTEGRATION.md shows the
 * stub a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes; host buffers are caller-owned, C-contiguous
 *     float64 (numpy); device memory is owned by the library.
 *   - every call returns 0 (EB_OK) or a negative eb_status; eb_last_error()
 *     gives the message.  Nothing throws across the boundary.
 *   - one host thread per context; calls are synchronous at return.
 *   - there is no CPU fallback: without a CUDA device eb_create fails.
 */
#ifndef EMCEE_B200_H
#define EMCEE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EB_ABI_VERSION 2

typedef enum eb_status {
  EB_OK = 0,
  EB_ERR_INVALID = -1,      /* bad argument / shape            -> ValueError  */
  EB_ERR_CUDA = -2,         /* CUDA runtime failure            -> RuntimeError */
  EB_ERR_COMM = -3,         /* NCCL / peer-memory failure      -> RuntimeError */
  EB_ERR_STATE = -4,        /* call order (no model, no state) -> RuntimeError */
  EB_ERR_UNSUPPORTED = -5,  /*                                 -> NotImplementedError */
  /* device-detected conditions the reference raises as exceptions */
  EB_ERR_NAN_LOGPROB = -10, /* ensemble.py:550-551 "Probability function returned NaN" */
  EB_ERR_INF_PARAM = -11,   /* ensemble.py:476-477 "At least one parameter value was infinite" */
  EB_ERR_NAN_PARAM = -12,   /* ensemble.py:478-479 "At least one parameter value was NaN" */
  EB_ERR_FEW_WALKERS = -13, /* moves/red_blue.py:64-70 RuntimeError (nwalkers < 2*ndim) */
  EB_ERR_NAN_INITIAL = -14  /* ensemble.py:357-358 "The initial log_prob was NaN" */
} eb_status;

/* registered device-side log-probability models (replace the Python callable
 * log_prob_fn of ensemble.py:79-83 / _FunctionWrapper ensemble.py:626-650) */
typedef enum eb_model_kind {
  EB_MODEL_GAUSS_ISO = 0,   /* -0.5*sum(x^2); params: none                                    */
  EB_MODEL_GAUSS_DENSE = 1, /* -0.5*(x-mu)^T A (x-mu); params: mu[D] then A[D*D] row-major    */
  EB_MODEL_ROSENBROCK = 2,  /* -sum b(x[i+1]-x[i]^2)^2+(a-x[i])^2; params: a, b               */
  EB_MODEL_RING = 3         /* -(|x|-R)^2/(2 s^2); params: R, s                               */
} eb_model_kind;

/* red-blue moves (moves/stretch.py, moves/de.py, moves/de_snooker.py) */
typedef enum eb_move_kind {
  EB_MOVE_STRETCH = 0, /* p0 = a        (stretch.py:22)                         */
  EB_MOVE_DE = 1,      /* p0 = sigma, p1 = gamma0 or NaN for 2.38/sqrt(2 ndim) (de.py:28,33-38) */
  EB_MOVE_SNOOKER = 2, /* p0 = gammas   (de_snooker.py:26); nsplits must be 4 (:28) */
  EB_MOVE_WALK = 3,    /* p0 = s, the number of helper walkers, or NaN for the whole complement (walk.py:24,32) */
  EB_MOVE_GAUSSIAN = 4 /* MHMove with a Gaussian proposal (mh.py:35-65, gaussian.py:32-119): `mode`, p1 = factor
                          or NaN, `cov`/`ncov` = the cov argument (1 scalar, ndim vector, ndim*ndim matrix);
                          not a red-blue move: nsplits / randomize_split are ignored */
} eb_move_kind;

typedef enum eb_gaussian_mode { /* gaussian.py:63,99-104 */
  EB_GAUSS_VECTOR = 0, EB_GAUSS_RANDOM = 1, EB_GAUSS_SEQUENTIAL = 2
} eb_gaussian_mode;

/* one entry of the move schedule (ensemble.py:115-129) with the RedBlueMove
 * constructor arguments (moves/red_blue.py:37-42) */
typedef struct eb_move {
  int32_t kind;             /* eb_move_kind */
  int32_t nsplits;          /* red_blue.py:40 */
  int32_t randomize_split;  /* red_blue.py:42 */
  int32_t live_dangerously; /* red_blue.py:41 */
  double weight;            /* un-normalised; normalised as ensemble.py:128-129 */
  double p0;
  double p1;
  /* ABI 2: GaussianMove only (zero / NULL otherwise) */
  int32_t mode;             /* eb_gaussian_mode */
  int32_t reserved;
  int64_t seq_index;        /* mode "sequential": the proposal's `index` (gaussian.py:64) when the call starts */
  const double* cov;        /* host pointer, read during the call */
  uint64_t ncov;
} eb_move;

typedef struct eb_ctx eb_ctx;

/* ---- lifetime ---------------------------------------------------------- */
int eb_abi_version(void);
/* number of visible CUDA devices (0 when the driver is absent). */
int eb_device_count(void);
/* replaces EnsembleSampler.__init__'s state set-up (ensemble.py:131-167): an
 * engine for an [nwalkers, ndim] float64 ensemble on CUDA device `device`, its
 * Philox key = seed, step counter = 0. */
int eb_create(int device, int64_t nwalkers, int64_t ndim, uint64_t seed, eb_ctx** out);
int eb_destroy(eb_ctx* ctx);
/* message of the last failing call on ctx (ctx == NULL: last eb_create failure
 * of this thread).  Pointer valid until the next call on the same ctx. */
const char* eb_last_error(const eb_ctx* ctx);

/* ---- model ------------------------------------------------------------- */
/* replaces passing log_prob_fn/args/kwargs (ensemble.py:79-98,169-171). */
int eb_model_set(eb_ctx* ctx, int kind, const double* params, size_t nparams);

/* ---- state (state.py:10-45) ------------------------------------------- */
/* State(initial_state, copy=True) + the initial compute_log_prob
 * (ensemble.py:312,350-358): copies coords[nwalkers*ndim] to the device;
 * log_prob == NULL -> evaluated on the device.  Non-finite coords / NaN
 * log-prob give the reference's errors. */
int eb_set_state(eb_ctx* ctx, const double* coords, const double* log_prob);
/* device -> host copy of the live state; either pointer may be NULL.
 * Sharded ensembles (after eb_comm_init): eb_set_state reads only the rows this
 * rank owns from the (globally indexed) host arrays, and eb_get_state returns
 * the GLOBAL state -- it replicates the other ranks' rows first and is
 * therefore COLLECTIVE (every rank calls it at the same point), as are
 * eb_get_naccepted, eb_step with accepted_last != NULL and eb_step_store. */
int eb_get_state(eb_ctx* ctx, double* coords, double* log_prob);
/* rows [row0, row0 + nrows) this context owns: the whole ensemble on one GPU,
 * the rank's row block after eb_comm_init. */
int eb_owned_rows(const eb_ctx* ctx, int64_t* row0, int64_t* nrows);
/* device -> host copy of rows [row0, row0 + nrows) of the live state into
 * coords[nrows * ndim] / log_prob[nrows] (either may be NULL).  Not collective:
 * on a sharded ensemble only the owned block (or any rows after a collective
 * read) is valid; other rows are refused with EB_ERR_STATE. */
int eb_get_state_rows(eb_ctx* ctx, int64_t row0, int64_t nrows, double* coords, double* log_prob);

/* ---- log-probability (ensemble.py:458-553) ------------------------------ */
/* EnsembleSampler.compute_log_prob(coords[m, ndim]) -> out[m], with the
 * isinf/isnan guards on the input (:476-479) and the NaN guard on the output
 * (:550-551). */
int eb_compute_log_prob(eb_ctx* ctx, const double* coords, size_t m, double* out);

/* ---- random state (ensemble.py:216-238) --------------------------------- */
/* The engine's "random_state" is (seed, step): every draw is a pure function
 * of (seed, step, split, active rank, purpose) -- see DESIGN.md "Draw
 * specification". */
int eb_set_rng(eb_ctx* ctx, uint64_t seed, uint64_t step);
int eb_get_rng(const eb_ctx* ctx, uint64_t* seed, uint64_t* step);

/* ---- the hot path ------------------------------------------------------- */
/* nsteps iterations of the sample() inner loop (ensemble.py:403-419): per step
 * draw one move from the schedule (:406), then Move.propose = the RedBlueMove
 * split cycle (moves/red_blue.py:52-106): split assignment (:76-80), per split
 * proposal (stretch.py:26-33 / de.py:40-64 / de_snooker.py:31-46), log-prob of
 * the proposals (:93), Metropolis accept (:96-101) and in-place update
 * (:103-104 -> moves/move.py:29-34).  accepted_last (nullable, nwalkers bytes)
 * receives the accept mask of the last step (the `accepted` propose returns).
 * Per-walker accept counts accumulate on the device (backend.py:229). */
int eb_step(eb_ctx* ctx, const eb_move* moves, size_t nmoves, uint64_t nsteps,
            uint8_t* accepted_last);
/* like eb_step with store=True (ensemble.py:416-417 -> backend.py:214-231):
 * every thin_by-th step's coords / log_prob are appended to the host arrays
 * chain[nstore, nwalkers, ndim], log_prob[nstore, nwalkers] (nstore =
 * nsteps / thin_by) and accepted[nwalkers] (float64, backend.py:31) is
 * incremented per accepted proposal of the stored steps' windows. */
int eb_step_store(eb_ctx* ctx, const eb_move* moves, size_t nmoves, uint64_t nsteps,
                  uint64_t thin_by, double* chain, double* log_prob, double* accepted);
/* per-walker number of accepted proposals since creation / eb_reset_counters
 * (numerator of acceptance_fraction, ensemble.py:555-558). */
int eb_get_naccepted(eb_ctx* ctx, uint64_t* naccepted);
/* how many steps of the LAST eb_step / eb_step_store call ran each entry of its move schedule
 * (picks[nmoves]): the host mirror of a stateful move (GaussianMove mode "sequential",
 * gaussian.py:102-103) advances its index by this count. */
int eb_move_picks(const eb_ctx* ctx, uint64_t* picks, size_t nmoves);
int eb_reset_counters(eb_ctx* ctx);

/* ---- chain analysis on the device --------------------------------------- */
/* Running moments of the chain for store=False runs (ensemble.py:287-291 keeps
 * nothing; a caller who wants the chain mean / covariance would otherwise need
 * a D2H of the state every step).  Enabled by eb_set_option("moments_every", n):
 * after every n-th step the rows this context owns are folded into device
 * accumulators (sum and outer-product sum on the FP64 tensor pipe).  Returns
 * mean[ndim], cov[ndim*ndim] (= np.mean / np.cov(rowvar=False, ddof=1) over
 * the accumulated (step, walker) samples), their number, and the total number
 * of accepted proposals of the owned walkers; any output may be NULL.  On a
 * sharded ensemble the values are per rank (the host combines them). */
int eb_moments(eb_ctx* ctx, double* mean, double* cov, uint64_t* count, uint64_t* naccepted_total);
/* walkers_independent (ensemble.py:653-663) on the device: gram[ndim*ndim] =
 * C^T C of the centred, column-normalised coords[rows, ndim] (:656-661), whose
 * extreme eigenvalues give cond(C)^2.  *flags: bit 0 = non-finite coordinate
 * (:655), bit 1 = a column with zero span (:659-660).  The D x D symmetric
 * eigen-solve stays on the host (numpy). */
int eb_walkers_gram(eb_ctx* ctx, const double* coords, size_t rows, double* gram, int* flags);
/* The device part of autocorr.integrated_time (autocorr.py:49-123, called from
 * backends/backend.py:130-150 on the stored chain): for chain[n_step, n_walker,
 * n_param] (host, C order) acf[n_param, n_step] = the walker average of the
 * normalised autocorrelation functions function_1d(chain[:, k, d])
 * (autocorr.py:21-46: FFT of the mean-subtracted series zero-padded to
 * 2*next_pow_two(n_step), power spectrum, inverse FFT, / acf[0]; :101-106).
 * Sokal's window search on acf (:107-109) is O(n_step * n_param) and stays
 * on the host.  Independent of the context's ensemble shape. */
int eb_autocorr(eb_ctx* ctx, const double* chain, size_t n_step, size_t n_walker, size_t n_param, double* acf);

/* ---- measurement / test taps ------------------------------------------- */
/* device time (ms, CUDA events on the engine's stream) of the last eb_step /
 * eb_step_store call, first launch to last, and the number of kernels it
 * launched. */
int eb_last_step_timing(const eb_ctx* ctx, double* ms, uint64_t* launches);
/* draws of the LAST half-step executed (known-answer tests): for each active
 * rank i of that split, partner walker ids (up to 3 per walker: stretch uses
 * [0]; DE [0]=p0,[1]=p1; snooker z,z1,z2), the proposal scalar (stretch zz,
 * DE gamma, snooker |s-z|) and the accept uniform.  Arrays sized nwalkers
 * (x3 for partners); *nactive returns the count. */
int eb_debug_taps(eb_ctx* ctx, int64_t* partners, double* scalar, double* u_accept,
                  int64_t* active, int64_t* nactive);
/* launch shape of the LAST fused red-blue half-step (test hook: which kernel
 * variant ran), out[EB_LAUNCH_CONFIG_FIELDS] = { kernel (0 none yet, 1 generic,
 * 2 tma_rows, 3 dense_dmma), walkers per tile (tma_rows, dense_dmma) or lanes
 * per walker (generic), elements per lane of the tma_rows register path (8, or
 * 0 for the run-time path), own row in registers (tma_rows, 0/1), warps per CTA
 * (dense_dmma: consumer warps), threads per CTA, CTAs, tiles of the half-step
 * (generic: active walkers) }.  n < EB_LAUNCH_CONFIG_FIELDS -> EB_ERR_INVALID. */
#define EB_LAUNCH_CONFIG_FIELDS 8
int eb_debug_launch_config(const eb_ctx* ctx, int64_t* out, size_t n);
/* per-tile cycle stamps of the dense_dmma consumers during the LAST half-step
 * launched (option "dmma_timeline"): [SM][8 consumers][8 tiles][6 events]. */
int eb_debug_timeline(eb_ctx* ctx, int64_t* out, size_t capacity, size_t* written);
/* engine options: "debug_taps" (0/1: record the draws of each half-step for
 * eb_debug_taps; forces the generic kernel), "dense_dmma" (0/1: allow the
 * FP64 tensor-core kernel for stretch + gauss_dense; default 1), "tma_rows" (0/1/2: the TMA row-gather kernel
 * for the HBM-bound models: off / rows short enough for several walkers per tile / any even ndim; default 2), "dmma_stagger" (0/1: staggered
 * first tiles at launch start; default 1), "dmma_group" (n >= 1: half-steps
 * fused into one persistent cooperative launch of that kernel, separated by an
 * in-kernel grid barrier -- and, on a P2P-sharded ensemble, a peer-flag barrier; default 1), "pdl" (0/1/2: consecutive dense_dmma launches chain as programmatic
 * dependent launches so a launch's prologue overlaps its predecessor's tail; 1 = on one GPU (default), 2 = on sharded ensembles too), "tma_own_reg" (0/1: tma_rows with the stretch move and rows of at most 512 bytes keeps the own row
 * in registers and stages only the partner rows; default 1), "dmma_local_first" (0/1/2: sharded dense_dmma -- build the first round of tiles from walkers whose
 * partner is local and take the peer barrier behind them; 0 never (default: the measured effect changes sign with the
 * number of GPUs), 1 when a consumer warp has at most two tiles per half-step, 2 always), "moments_every" (n >= 0: see
 * eb_moments; setting it resets the accumulators), "dmma_timeline" (0/1: record consumer cycle stamps
 * for eb_debug_timeline), "grid_cap" (n >= 0: at most n CTAs for the grid-strided launches sized by the SM count --
 * the tma_rows and dense_dmma half-steps and the dense_dmma log-probability -- so each warp works through more
 * tiles; results do not depend on it (draws are keyed by active rank, tiles are dealt by stride); 0 = no cap,
 * the default), "l2_flush"
 * (0/1: benchmark hygiene -- write a 256 MiB buffer before every step and time
 * each step with its own CUDA-event pair, so eb_last_step_timing excludes the
 * flush). */
int eb_set_option(eb_ctx* ctx, const char* name, int64_t value);
/* name of the kernel variant the last eb_step used for its half-steps
 * ("generic", "dense_dmma", ...). */
const char* eb_last_kernel_name(const eb_ctx* ctx);

/* device micro-benchmarks that anchor the FP64 roofline (MEASURED_PEAKS.json has
 * only HBM and bf16 peaks): what = 0 DFMA, 1 DMMA m8n8k4, 2 DMMA m16n8k8,
 * 3 DMMA m16n8k16 (result in TFLOP/s), 4 HBM copy (GB/s).  Current device. */
int eb_microbench(int what, int warps_per_sm, double* result);
/* page-locked host memory for callers that want full-speed H2D/D2H of the
 * arrays they hand to eb_set_state / eb_get_state / eb_step_store. */
int eb_host_alloc(size_t bytes, void** out);
int eb_host_free(void* ptr);

/* ---- multi-GPU: one process per GPU, walkers sharded by row block ------- */
#define EB_COMM_ID_BYTES 128
/* rank 0 creates the id (ncclGetUniqueId), the host side broadcasts it. */
int eb_comm_id(char id[EB_COMM_ID_BYTES]);
/* join the communicator.  After this, nwalkers is the GLOBAL ensemble size,
 * rank r owns walkers [r*N/R, (r+1)*N/R) and eb_step exchanges the updated
 * rows after every split (one ncclAllGather, or peer-memory loads when
 * mode == EB_COMM_P2P). */
#define EB_COMM_ALLGATHER 0
#define EB_COMM_P2P 1
int eb_comm_init(eb_ctx* ctx, const char id[EB_COMM_ID_BYTES], int rank, int nranks, int mode);
/* peer-memory set-up for EB_COMM_P2P: export this rank's handles, then import
 * all ranks' (the host side all-gathers the blobs between the two calls). */
#define EB_IPC_BLOB_BYTES 256
int eb_comm_export(eb_ctx* ctx, char blob[EB_IPC_BLOB_BYTES]);
int eb_comm_import(eb_ctx* ctx, const char* blobs /* nranks * EB_IPC_BLOB_BYTES */);

/* measurement: GB/s of reading rank `peer`'s walker array (own rank = local HBM) with
 * what = 0 streaming 16-byte loads, 1 random whole rows (16-byte loads), 2 random whole rows
 * through TMA bulk copies (the dense_dmma producers' pattern). */
int eb_comm_probe(eb_ctx* ctx, int peer, int what, double* gbs);

#ifdef __cplusplus
}
#endif
#endif /* EMCEE_B200_H */
