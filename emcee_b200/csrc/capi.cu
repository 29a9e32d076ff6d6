// C ABI of the engine (include/emcee_b200.h): context, host-side step loop,
// state / model transfer, error mapping.  No torch, no CPU fallback.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "comm.h"
#include "engine.cuh"

using namespace eb;

struct eb_ctx {
  int device = 0;
  int sm_count = 0;
  int64_t N = 0;
  int D = 0;
  uint64_t seed = 0, step = 0;
  cudaStream_t st = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;

  double* coords = nullptr;
  double* logp = nullptr;
  uint8_t* accepted = nullptr;
  unsigned long long* nacc = nullptr;
  int* status_dev = nullptr;
  int* status_host = nullptr;  // pinned

  ModelDev model{};
  double* model_params = nullptr;
  double* model_chol = nullptr;
  bool have_model = false, have_state = false;

  int32_t* order = nullptr;  // [table_cap, N]
  size_t table_cap = 0;
  StepInfo* info_dev = nullptr;
  StepInfo* info_host = nullptr;  // pinned
  HalfDesc* descs_dev = nullptr;  // [table_cap * MAX_SPLITS] half-step descriptors of a chunk (dense_dmma)
  HalfDesc* descs_host = nullptr;  // pinned
  unsigned long long* gbar = nullptr;  // grid-barrier counter of the persistent dense_dmma kernel
  unsigned long long gbar_count = 0;   // arrivals issued so far
  // split tables already on the device: steps [tbl_step0, tbl_step0 + tbl_n) of key tbl_seed, built with tbl_info
  uint64_t tbl_seed = 0, tbl_step0 = 0;
  size_t tbl_n = 0;
  std::vector<StepInfo> tbl_info;

  double* scratch_x = nullptr;
  double* scratch_lp = nullptr;
  size_t scratch_rows = 0;

  // pinned staging for eb_step_store
  double* stage[2] = {nullptr, nullptr};
  uint8_t* stage_acc[2] = {nullptr, nullptr};
  cudaEvent_t stage_ev[2] = {nullptr, nullptr};

  bool debug = false;
  int64_t* tap_partners = nullptr;
  double* tap_scalar = nullptr;
  double* tap_u = nullptr;
  int64_t* tap_active = nullptr;
  int64_t tap_count = 0;
  long long* timeline = nullptr;  // dense_dmma instrumentation buffer (option "dmma_timeline")

  // optional L2 flush between steps (benchmark hygiene): per-step event pairs
  bool l2_flush = false;
  void* flush_buf = nullptr;
  size_t flush_bytes = (size_t)256 << 20;
  std::vector<cudaEvent_t> ev_pool;

  double last_ms = 0.0;
  uint64_t last_launches = 0;
  const char* last_kernel = "none";
  bool allow_dmma = true;
  int allow_tma = 2;  // TMA row-gather kernel for the HBM-bound models: 0 off, 1 short rows only, 2 long rows too
  bool tma_own_reg = true;  // tma_rows, stretch rows <= 512 B: own rows through registers instead of the TMA unit
  bool fused_last = false;  // the last dense_dmma launch carried the P2P barrier itself
  int dmma_stagger = 1;
  int dmma_group = 1;  // half-steps per persistent dense_dmma launch (1: a launch per half-step)
  int pdl = 1;           // dense_dmma launches chain as programmatic dependents (1: one GPU only, 2: sharded too)
  int grid_cap = 0;      // most CTAs of the grid-strided half-step / dense log-prob launches (0: no cap)
  LaunchShape last_shape{};  // launch shape of the last fused half-step (eb_debug_launch_config)
  int local_first = 0;  // sharded dense_dmma: local-partner tiles first, peer barrier behind them (0 never, 1 auto, 2 always)
  bool chain_ok = false; // the last operation enqueued on the stream is a dense_dmma kernel of this run
  // multi-GPU: log_prob / accept mask / counters (and, P2P, coords) of rows owned by OTHER ranks are stale
  // on this rank until the next collective read (eb_get_state, eb_get_naccepted, ...) replicates them
  bool replicas_dirty = false;

  // running chain moments (eb_moments): sum of (x - shift) and of its outer product over the owned
  // rows of every `moments_every`-th step
  uint64_t moments_every = 0;
  double* mom_acc = nullptr;      // [D + D*D] accumulators
  double* mom_shift = nullptr;    // [D]
  double* mom_partial = nullptr;  // per-CTA partials of one accumulation
  unsigned long long mom_count = 0;
  bool mom_have_shift = false;

  // WalkMove / GaussianMove scratch (moves_extra.cu)
  double* qbuf = nullptr;       // [N, D] proposals
  double* walk_work = nullptr;  // [D shift | D + D*D moment sums | D*D cov | D*D L]
  double* gauss_dev = nullptr;  // per schedule entry: scale / factor L of GaussianMove
  size_t gauss_cap = 0;
  std::vector<uint64_t> picks;  // per schedule entry: steps of the last call that ran it

  Comm comm;  // multi-GPU (comm.h)

  std::string err;
};

static thread_local std::string g_create_err;

#define FAIL(ctx, code, ...)                      \
  do {                                            \
    char _b[512];                                 \
    snprintf(_b, sizeof(_b), __VA_ARGS__);        \
    (ctx)->err = _b;                              \
    return (code);                                \
  } while (0)

#define CK(ctx, call)                                                                      \
  do {                                                                                     \
    cudaError_t _e = (call);                                                               \
    if (_e != cudaSuccess) {                                                               \
      cudaGetLastError();                                                                  \
      FAIL(ctx, EB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, \
           __LINE__);                                                                      \
    }                                                                                      \
  } while (0)

// map (and clear) the device status word to the reference's exceptions, in the
// order compute_log_prob raises them (ensemble.py:476-479, 550-551)
static int check_status(eb_ctx* c) {
  const int f = *c->status_host;
  if (f == 0) return EB_OK;
  *c->status_host = 0;
  cudaMemsetAsync(c->status_dev, 0, sizeof(int), c->st);
  cudaStreamSynchronize(c->st);
  if (f & FLAG_COMM_TIMEOUT) FAIL(c, EB_ERR_COMM, "peer-memory barrier timed out: another rank did not arrive");
  if (f & FLAG_INF_PARAM) FAIL(c, EB_ERR_INF_PARAM, "At least one parameter value was infinite");
  if (f & FLAG_NAN_PARAM) FAIL(c, EB_ERR_NAN_PARAM, "At least one parameter value was NaN");
  FAIL(c, EB_ERR_NAN_LOGPROB, "Probability function returned NaN");
}

static int fetch_status(eb_ctx* c) {
  CK(c, cudaMemcpyAsync(c->status_host, c->status_dev, sizeof(int), cudaMemcpyDeviceToHost, c->st));
  CK(c, cudaStreamSynchronize(c->st));
  return check_status(c);
}

extern "C" {

int eb_abi_version(void) { return EB_ABI_VERSION; }

int eb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

const char* eb_last_error(const eb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int eb_create(int device, int64_t nwalkers, int64_t ndim, uint64_t seed, eb_ctx** out) {
  if (!out) return EB_ERR_INVALID;
  *out = nullptr;
  if (nwalkers < 2 || ndim < 1 || nwalkers > (int64_t)0x7fffffff || ndim > 16384) {
    g_create_err = "eb_create: need 2 <= nwalkers < 2^31 and 1 <= ndim <= 16384";
    return EB_ERR_INVALID;
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    g_create_err = std::string("eb_create: no CUDA device (") + cudaGetErrorString(e) +
                   "); this engine has no CPU fallback";
    return EB_ERR_CUDA;
  }
  if (device < 0 || device >= ndev) {
    g_create_err = "eb_create: device index out of range";
    return EB_ERR_INVALID;
  }
  eb_ctx* c = new eb_ctx();
  c->device = device;
  c->N = nwalkers;
  c->D = (int)ndim;
  c->seed = seed;
  if (const char* e = getenv("EMCEE_B200_TMA_ROWS")) c->allow_tma = atoi(e);  // developer override
  auto fail = [&](const char* what, cudaError_t err) {
    g_create_err = std::string("eb_create: ") + what + ": " + cudaGetErrorString(err);
    eb_destroy(c);
    return EB_ERR_CUDA;
  };
#define CC(call)                             \
  do {                                       \
    cudaError_t _e = (call);                 \
    if (_e != cudaSuccess) return fail(#call, _e); \
  } while (0)
  CC(cudaSetDevice(device));
  cudaDeviceProp prop;
  CC(cudaGetDeviceProperties(&prop, device));
  c->sm_count = prop.multiProcessorCount;
  CC(cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking));
  CC(cudaEventCreate(&c->ev0));
  CC(cudaEventCreate(&c->ev1));
  const size_t nd = (size_t)nwalkers * (size_t)ndim;
  // the tail holds the peer-memory barrier flags so one IPC handle exports both
  CC(cudaMalloc(&c->coords, nd * sizeof(double) + MAX_RANKS * sizeof(unsigned)));
  CC(cudaMalloc(&c->logp, (size_t)nwalkers * sizeof(double)));
  CC(cudaMalloc(&c->accepted, (size_t)nwalkers));
  CC(cudaMalloc(&c->nacc, (size_t)nwalkers * sizeof(unsigned long long)));
  CC(cudaMalloc(&c->status_dev, sizeof(int)));
  CC(cudaMallocHost(&c->status_host, sizeof(int)));
  *c->status_host = 0;
  CC(cudaMemsetAsync(c->status_dev, 0, sizeof(int), c->st));
  CC(cudaMemsetAsync(c->accepted, 0, (size_t)nwalkers, c->st));
  CC(cudaMemsetAsync(c->nacc, 0, (size_t)nwalkers * sizeof(unsigned long long), c->st));
  // split tables for a chunk of steps: <= 64 MiB, 1..512 steps
  size_t cap = (64u << 20) / ((size_t)nwalkers * sizeof(int32_t));
  cap = std::max<size_t>(1, std::min<size_t>(cap, 512));
  c->table_cap = cap;
  CC(cudaMalloc(&c->order, cap * (size_t)nwalkers * sizeof(int32_t)));
  CC(cudaMalloc(&c->info_dev, cap * sizeof(StepInfo)));
  CC(cudaMallocHost(&c->info_host, cap * sizeof(StepInfo)));
  CC(cudaMalloc(&c->descs_dev, cap * MAX_SPLITS * sizeof(HalfDesc)));
  CC(cudaMallocHost(&c->descs_host, cap * MAX_SPLITS * sizeof(HalfDesc)));
  CC(cudaMalloc(&c->gbar, sizeof(unsigned long long)));
  CC(cudaMemsetAsync(c->gbar, 0, sizeof(unsigned long long), c->st));
  CC(cudaStreamSynchronize(c->st));
#undef CC
  *out = c;
  return EB_OK;
}

int eb_destroy(eb_ctx* c) {
  if (!c) return EB_OK;
  cudaSetDevice(c->device);
  comm_destroy(c->comm);
  if (c->st) cudaStreamSynchronize(c->st);
  cudaFree(c->coords);
  cudaFree(c->logp);
  cudaFree(c->accepted);
  cudaFree(c->nacc);
  cudaFree(c->status_dev);
  cudaFreeHost(c->status_host);
  cudaFree(c->model_params);
  cudaFree(c->model_chol);
  cudaFree(c->order);
  cudaFree(c->info_dev);
  cudaFreeHost(c->info_host);
  cudaFree(c->descs_dev);
  cudaFreeHost(c->descs_host);
  cudaFree(c->gbar);
  cudaFree(c->scratch_x);
  cudaFree(c->scratch_lp);
  for (int k = 0; k < 2; ++k) {
    cudaFreeHost(c->stage[k]);
    cudaFreeHost(c->stage_acc[k]);
    if (c->stage_ev[k]) cudaEventDestroy(c->stage_ev[k]);
  }
  cudaFree(c->flush_buf);
  cudaFree(c->qbuf);
  cudaFree(c->walk_work);
  cudaFree(c->gauss_dev);
  cudaFree(c->mom_acc);
  cudaFree(c->mom_shift);
  cudaFree(c->mom_partial);
  for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
  cudaFree(c->timeline);
  cudaFree(c->tap_partners);
  cudaFree(c->tap_scalar);
  cudaFree(c->tap_u);
  cudaFree(c->tap_active);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->st) cudaStreamDestroy(c->st);
  cudaGetLastError();
  delete c;
  return EB_OK;
}

// ---- model -----------------------------------------------------------------
// Lower Cholesky factor of the symmetric part of A, packed for the DMMA kernel
// (dense_dmma.cu).  Returns false when A is not numerically positive definite.
static bool cholesky_lower(const double* A, int D, std::vector<double>& L) {
  L.assign((size_t)D * D, 0.0);
  for (int j = 0; j < D; ++j) {
    double d = 0.5 * (A[(size_t)j * D + j] + A[(size_t)j * D + j]);
    for (int k = 0; k < j; ++k) d -= L[(size_t)j * D + k] * L[(size_t)j * D + k];
    if (!(d > 0.0) || !isfinite(d)) return false;
    const double ljj = sqrt(d);
    L[(size_t)j * D + j] = ljj;
    for (int i = j + 1; i < D; ++i) {
      double s = 0.5 * (A[(size_t)i * D + j] + A[(size_t)j * D + i]);
      for (int k = 0; k < j; ++k) s -= L[(size_t)i * D + k] * L[(size_t)j * D + k];
      L[(size_t)i * D + j] = s / ljj;
    }
  }
  return true;
}

int eb_model_set(eb_ctx* c, int kind, const double* params, size_t nparams) {
  if (!c) return EB_ERR_INVALID;
  CK(c, cudaSetDevice(c->device));
  const size_t D = (size_t)c->D;
  ModelDev m{};
  m.kind = kind;
  std::vector<double> host;
  switch (kind) {
    case EB_MODEL_GAUSS_ISO:
      if (nparams != 0) FAIL(c, EB_ERR_INVALID, "gauss_iso takes no parameters");
      break;
    case EB_MODEL_GAUSS_DENSE:
      if (nparams != D + D * D || !params)
        FAIL(c, EB_ERR_INVALID, "gauss_dense takes mu[D] followed by A[D*D] (got %zu doubles)", nparams);
      for (size_t k = 0; k < nparams; ++k)
        if (!isfinite(params[k])) FAIL(c, EB_ERR_INVALID, "gauss_dense parameters must be finite");
      host.assign(params, params + nparams);
      for (size_t k = 0; k < D; ++k)
        if (params[k] != 0.0) m.s0 = 1.0;  // non-zero mean (dense_dmma.cu picks its variant by this)
      break;
    case EB_MODEL_ROSENBROCK:
    case EB_MODEL_RING:
      if (nparams != 2 || !params) FAIL(c, EB_ERR_INVALID, "model takes exactly 2 parameters");
      if (kind == EB_MODEL_RING && !(params[1] > 0.0)) FAIL(c, EB_ERR_INVALID, "ring sigma must be > 0");
      if (kind == EB_MODEL_ROSENBROCK && D < 2) FAIL(c, EB_ERR_INVALID, "rosenbrock needs ndim >= 2");
      m.s0 = params[0];
      m.s1 = params[1];
      break;
    default:
      FAIL(c, EB_ERR_INVALID, "unknown model kind %d", kind);
  }
  CK(c, cudaStreamSynchronize(c->st));
  cudaFree(c->model_params);
  cudaFree(c->model_chol);
  c->model_params = nullptr;
  c->model_chol = nullptr;
  if (!host.empty()) {
    CK(c, cudaMalloc(&c->model_params, host.size() * sizeof(double)));
    CK(c, cudaMemcpy(c->model_params, host.data(), host.size() * sizeof(double), cudaMemcpyHostToDevice));
    m.params = c->model_params;
    if (kind == EB_MODEL_GAUSS_DENSE && dense_dmma_supported(c->D)) {
      std::vector<double> L;
      if (cholesky_lower(host.data() + D, c->D, L)) {
        std::vector<double> packed(dense_dmma_factor_doubles(c->D));
        dense_dmma_pack_factor(L.data(), c->D, packed.data());
        CK(c, cudaMalloc(&c->model_chol, packed.size() * sizeof(double)));
        CK(c, cudaMemcpy(c->model_chol, packed.data(), packed.size() * sizeof(double),
                         cudaMemcpyHostToDevice));
        m.chol = c->model_chol;
      }
    }
  }
  c->model = m;
  c->have_model = true;
  return EB_OK;
}

// CTA count of a grid-strided launch sized `full` (a multiple of the SM count), under option "grid_cap"
static int capped_grid(const eb_ctx* c, int full) { return c->grid_cap > 0 && c->grid_cap < full ? c->grid_cap : full; }

// ---- log-prob ----------------------------------------------------------------
// rows of x -> out with the kernel that matches the stepping path of the model
static cudaError_t launch_logprob(eb_ctx* c, const double* x, int64_t rows, double* out) {
  if (c->allow_dmma && c->model.kind == EB_MODEL_GAUSS_DENSE && c->model.chol != nullptr)
    return launch_logprob_dense_dmma(c->model, c->D, x, rows, out, c->status_dev, capped_grid(c, 2 * c->sm_count),
                                     c->st);
  return launch_logprob_generic(c->model, x, rows, c->D, out, c->status_dev, c->st);
}

static int ensure_scratch(eb_ctx* c, size_t rows) {
  if (rows <= c->scratch_rows) return EB_OK;
  CK(c, cudaStreamSynchronize(c->st));
  cudaFree(c->scratch_x);
  cudaFree(c->scratch_lp);
  c->scratch_x = nullptr;
  c->scratch_lp = nullptr;
  c->scratch_rows = 0;
  CK(c, cudaMalloc(&c->scratch_x, rows * (size_t)c->D * sizeof(double)));
  CK(c, cudaMalloc(&c->scratch_lp, rows * sizeof(double)));
  c->scratch_rows = rows;
  return EB_OK;
}

int eb_compute_log_prob(eb_ctx* c, const double* coords, size_t m, double* out) {
  if (!c) return EB_ERR_INVALID;
  if (!c->have_model) FAIL(c, EB_ERR_STATE, "eb_compute_log_prob: no model set");
  if (m == 0) return EB_OK;
  if (!coords || !out) FAIL(c, EB_ERR_INVALID, "eb_compute_log_prob: null buffer");
  CK(c, cudaSetDevice(c->device));
  int rc = ensure_scratch(c, m);
  if (rc) return rc;
  CK(c, cudaMemcpyAsync(c->scratch_x, coords, m * (size_t)c->D * sizeof(double), cudaMemcpyHostToDevice,
                        c->st));
  CK(c, launch_logprob(c, c->scratch_x, (int64_t)m, c->scratch_lp));
  CK(c, cudaMemcpyAsync(out, c->scratch_lp, m * sizeof(double), cudaMemcpyDeviceToHost, c->st));
  return fetch_status(c);
}

// ---- state -------------------------------------------------------------------
// rows [r0, r1) this context owns (the whole ensemble on one GPU)
static void owned_rows(const eb_ctx* c, int64_t& r0, int64_t& r1) {
  r0 = 0;
  r1 = c->N;
  if (c->comm.nranks > 1) {
    r0 = c->comm.rows_per_rank * c->comm.rank;
    r1 = r0 + c->comm.rows_per_rank;
  }
}

// multi-GPU: make log_prob / accept mask / counters (and coords in P2P mode) of every rank's rows
// valid on this rank.  COLLECTIVE: every rank calls it at the same point (the Python layer does).
static int sync_replicas(eb_ctx* c) {
  if (c->comm.nranks == 1 || !c->replicas_dirty) return EB_OK;
  uint64_t launches = 0;
  c->chain_ok = false;
  if (comm_sync_state(c->comm, c->st, c->status_dev, c->logp, c->accepted, c->nacc, launches))
    FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
  c->fused_last = false;
  CK(c, cudaStreamSynchronize(c->st));
  c->replicas_dirty = false;
  return EB_OK;
}

int eb_set_state(eb_ctx* c, const double* coords, const double* log_prob) {
  if (!c) return EB_ERR_INVALID;
  if (!coords) FAIL(c, EB_ERR_INVALID, "eb_set_state: coords is null");
  if (!c->have_model) FAIL(c, EB_ERR_STATE, "eb_set_state: no model set");
  CK(c, cudaSetDevice(c->device));
  const size_t D = (size_t)c->D;
  c->have_state = false;
  c->chain_ok = false;
  if (log_prob) {
    for (int64_t w = 0; w < c->N; ++w)
      if (isnan(log_prob[w])) FAIL(c, EB_ERR_NAN_INITIAL, "The initial log_prob was NaN");  // ensemble.py:357-358
  }
  // Sharded ensembles: only the rows this rank owns cross PCIe (the host arrays are still indexed by
  // global walker id); non-owned rows are never read by the kernels in P2P mode and are filled by one
  // all-gather in EB_COMM_ALLGATHER mode.
  int64_t r0, r1;
  owned_rows(c, r0, r1);
  const size_t rows = (size_t)(r1 - r0);
  uint64_t launches = 0;
  if (c->comm.nranks > 1 && c->comm.mode == EB_COMM_P2P && c->comm.imported) {
    // no peer may still be pulling the rows that are about to be overwritten
    if (comm_barrier(c->comm, c->st, c->status_dev, launches)) FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
    c->fused_last = false;
  }
  CK(c, cudaMemcpyAsync(c->coords + (size_t)r0 * D, coords + (size_t)r0 * D, rows * D * sizeof(double),
                        cudaMemcpyHostToDevice, c->st));
  if (log_prob) {
    CK(c, cudaMemcpyAsync(c->logp + r0, log_prob + r0, rows * sizeof(double), cudaMemcpyHostToDevice, c->st));
  } else {
    CK(c, launch_logprob(c, c->coords + (size_t)r0 * D, (int64_t)rows, c->logp + r0));
  }
  if (c->comm.nranks > 1) {
    if (c->comm.mode == EB_COMM_ALLGATHER && comm_gather_coords(c->comm, c->st, launches))
      FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
    if (c->comm.mode == EB_COMM_P2P && c->comm.imported &&
        comm_barrier(c->comm, c->st, c->status_dev, launches))  // every rank's block is in place
      FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
    c->replicas_dirty = true;
  }
  int rc = fetch_status(c);
  if (rc) return rc;
  c->have_state = true;
  return EB_OK;
}

int eb_get_state(eb_ctx* c, double* coords, double* log_prob) {
  if (!c) return EB_ERR_INVALID;
  if (!c->have_state) FAIL(c, EB_ERR_STATE, "eb_get_state: no state set");
  CK(c, cudaSetDevice(c->device));
  int rc = sync_replicas(c);  // multi-GPU: the GLOBAL state (collective)
  if (rc) return rc;
  c->chain_ok = false;
  if (coords)
    CK(c, cudaMemcpyAsync(coords, c->coords, (size_t)c->N * c->D * sizeof(double), cudaMemcpyDeviceToHost,
                          c->st));
  if (log_prob)
    CK(c, cudaMemcpyAsync(log_prob, c->logp, (size_t)c->N * sizeof(double), cudaMemcpyDeviceToHost, c->st));
  CK(c, cudaStreamSynchronize(c->st));
  return EB_OK;
}

int eb_owned_rows(const eb_ctx* c, int64_t* row0, int64_t* nrows) {
  if (!c) return EB_ERR_INVALID;
  int64_t r0, r1;
  owned_rows(c, r0, r1);
  if (row0) *row0 = r0;
  if (nrows) *nrows = r1 - r0;
  return EB_OK;
}

int eb_get_state_rows(eb_ctx* c, int64_t row0, int64_t nrows, double* coords, double* log_prob) {
  if (!c) return EB_ERR_INVALID;
  if (!c->have_state) FAIL(c, EB_ERR_STATE, "eb_get_state_rows: no state set");
  if (row0 < 0 || nrows < 0 || row0 + nrows > c->N) FAIL(c, EB_ERR_INVALID, "eb_get_state_rows: rows out of range");
  int64_t r0, r1;
  owned_rows(c, r0, r1);
  if (c->replicas_dirty && (row0 < r0 || row0 + nrows > r1))
    FAIL(c, EB_ERR_STATE, "eb_get_state_rows: rows [%lld, %lld) are owned by another rank and not replicated here; "
         "read the owned block [%lld, %lld) or call eb_get_state (collective) first",
         (long long)row0, (long long)(row0 + nrows), (long long)r0, (long long)r1);
  CK(c, cudaSetDevice(c->device));
  c->chain_ok = false;
  if (coords && nrows)
    CK(c, cudaMemcpyAsync(coords, c->coords + (size_t)row0 * c->D, (size_t)nrows * c->D * sizeof(double),
                          cudaMemcpyDeviceToHost, c->st));
  if (log_prob && nrows)
    CK(c, cudaMemcpyAsync(log_prob, c->logp + row0, (size_t)nrows * sizeof(double), cudaMemcpyDeviceToHost, c->st));
  CK(c, cudaStreamSynchronize(c->st));
  return EB_OK;
}

int eb_set_rng(eb_ctx* c, uint64_t seed, uint64_t step) {
  if (!c) return EB_ERR_INVALID;
  c->seed = seed;
  c->step = step;
  return EB_OK;
}

int eb_get_rng(const eb_ctx* c, uint64_t* seed, uint64_t* step) {
  if (!c) return EB_ERR_INVALID;
  if (seed) *seed = c->seed;
  if (step) *step = c->step;
  return EB_OK;
}

}  // extern "C"

// ---- the hot path --------------------------------------------------------------
namespace {

struct Schedule {
  std::vector<eb_move> moves;
  std::vector<double> cdf;
  // GaussianMove: form (0 scalar, 1 diagonal, 2 full) and where its scale / Cholesky factor sits in gauss_dev
  std::vector<int> gform;
  std::vector<size_t> goff;
};

// thresholded lower Cholesky factor (the draw specification's multivariate_normal; oracle/philox.py chol_psd)
void chol_psd_host(const double* A, int D, std::vector<double>& L) {
  L.assign((size_t)D * D, 0.0);
  double m = 0.0;
  for (int j = 0; j < D; ++j) m = std::max(m, A[(size_t)j * D + j]);
  const double tol = 1e-12 * m;
  for (int j = 0; j < D; ++j) {
    double d = A[(size_t)j * D + j];
    for (int k = 0; k < j; ++k) d -= L[(size_t)j * D + k] * L[(size_t)j * D + k];
    if (!(d > tol)) continue;
    const double piv = sqrt(d);
    L[(size_t)j * D + j] = piv;
    for (int i = j + 1; i < D; ++i) {
      double v = A[(size_t)i * D + j];
      for (int k = 0; k < j; ++k) v -= L[(size_t)i * D + k] * L[(size_t)j * D + k];
      L[(size_t)i * D + j] = v / piv;
    }
  }
}

int build_schedule(eb_ctx* c, const eb_move* moves, size_t nmoves, Schedule& s) {
  if (!moves || nmoves == 0) FAIL(c, EB_ERR_INVALID, "eb_step: empty move schedule");
  s.moves.assign(moves, moves + nmoves);
  double tot = 0.0;
  s.gform.assign(nmoves, 0);
  s.goff.assign(nmoves, 0);
  std::vector<double> ghost;  // host image of gauss_dev
  for (size_t mi = 0; mi < nmoves; ++mi) {
    eb_move& m = s.moves[mi];
    if (m.kind < EB_MOVE_STRETCH || m.kind > EB_MOVE_GAUSSIAN)
      FAIL(c, EB_ERR_INVALID, "eb_step: unknown move kind %d", m.kind);
    if ((m.kind == EB_MOVE_WALK || m.kind == EB_MOVE_GAUSSIAN) && c->comm.nranks > 1)
      FAIL(c, EB_ERR_UNSUPPORTED, "eb_step: WalkMove / GaussianMove are not sharded across GPUs yet");
    if ((m.kind == EB_MOVE_WALK || m.kind == EB_MOVE_GAUSSIAN) && c->debug)
      FAIL(c, EB_ERR_UNSUPPORTED, "eb_step: debug taps do not cover WalkMove / GaussianMove");
    if (m.kind == EB_MOVE_GAUSSIAN) {
      const size_t D = (size_t)c->D;
      if (!m.cov || (m.ncov != 1 && m.ncov != D && m.ncov != D * D) || (D == 1 && m.ncov != 1))
        FAIL(c, EB_ERR_INVALID, "Invalid proposal scale dimensions");  // gaussian.py:53-54
      if (m.mode < EB_GAUSS_VECTOR || m.mode > EB_GAUSS_SEQUENTIAL)
        FAIL(c, EB_ERR_INVALID, "eb_step: unknown GaussianMove mode %d", m.mode);
      if (!isnan(m.p1) && m.p1 < 1.0) FAIL(c, EB_ERR_INVALID, "'factor' must be >= 1.0");  // gaussian.py:69-70
      if (!(m.weight >= 0.0) || !isfinite(m.weight)) FAIL(c, EB_ERR_INVALID, "eb_step: bad move weight");
      s.goff[mi] = ghost.size();
      if (m.ncov == D * D && D > 1) {
        if (m.mode != EB_GAUSS_VECTOR)
          FAIL(c, EB_ERR_INVALID, "a full proposal covariance only supports mode 'vector'");  // gaussian.py:110-111
        s.gform[mi] = 2;
        std::vector<double> L;
        chol_psd_host(m.cov, c->D, L);
        ghost.insert(ghost.end(), L.begin(), L.end());
        ghost.resize(ghost.size() + D);  // the shared shift v[D] of a step lives behind its factor
      } else {
        s.gform[mi] = m.ncov == 1 ? 0 : 1;
        for (size_t k = 0; k < m.ncov; ++k) {
          if (!(m.cov[k] >= 0.0)) FAIL(c, EB_ERR_INVALID, "GaussianMove: variances must be >= 0");
          ghost.push_back(sqrt(m.cov[k]));  // gaussian.py:45,58
        }
      }
      m.nsplits = 1;  // the split table of such a step is never read
      m.randomize_split = 0;
      tot += m.weight;
      continue;
    }
    if (m.kind == EB_MOVE_WALK && !isnan(m.p0)) {
      const int64_t nc_min = c->N - (c->N + m.nsplits - 1) / std::max(m.nsplits, 1);
      if (m.p0 != floor(m.p0) || m.p0 < 2 || (m.nsplits >= 2 && m.p0 > (double)nc_min))
        FAIL(c, EB_ERR_INVALID, "eb_step: WalkMove needs 2 <= s <= size of the smallest complement (got %g)", m.p0);
      if ((int64_t)m.p0 != nc_min && !walk_subset_supported(c->D, (int)m.p0))
        FAIL(c, EB_ERR_UNSUPPORTED, "eb_step: WalkMove with a helper subset is limited to ndim <= 64 and s <= 4096");
    }
    if (m.kind == EB_MOVE_WALK && c->D > 1024) FAIL(c, EB_ERR_UNSUPPORTED, "eb_step: WalkMove is limited to ndim <= 1024");
    if (m.nsplits < 2 || m.nsplits > MAX_SPLITS || m.nsplits > c->N)
      FAIL(c, EB_ERR_UNSUPPORTED, "eb_step: nsplits must be in [2, min(%d, nwalkers)] (got %d)", MAX_SPLITS,
           m.nsplits);
    if (m.kind == EB_MOVE_SNOOKER && m.nsplits != 4)
      FAIL(c, EB_ERR_INVALID, "eb_step: DESnookerMove uses nsplits = 4 (de_snooker.py:28)");
    if (m.kind == EB_MOVE_DE && c->N - (c->N + m.nsplits - 1) / m.nsplits < 2)
      FAIL(c, EB_ERR_INVALID, "eb_step: DEMove needs at least 2 complement walkers");
    if (!(m.weight >= 0.0) || !isfinite(m.weight)) FAIL(c, EB_ERR_INVALID, "eb_step: bad move weight");
    if (m.kind == EB_MOVE_STRETCH && !(m.p0 > 0.0)) FAIL(c, EB_ERR_INVALID, "eb_step: stretch scale a must be > 0");
    tot += m.weight;
  }
  if (!(tot > 0.0)) FAIL(c, EB_ERR_INVALID, "eb_step: move weights sum to zero");
  if (!ghost.empty()) {
    if (ghost.size() > c->gauss_cap) {
      CK(c, cudaStreamSynchronize(c->st));
      cudaFree(c->gauss_dev);
      c->gauss_dev = nullptr;
      c->gauss_cap = 0;
      CK(c, cudaMalloc(&c->gauss_dev, ghost.size() * sizeof(double)));
      c->gauss_cap = ghost.size();
    }
    CK(c, cudaMemcpyAsync(c->gauss_dev, ghost.data(), ghost.size() * sizeof(double), cudaMemcpyHostToDevice, c->st));
    CK(c, cudaStreamSynchronize(c->st));  // ghost is a local
  }
  c->picks.assign(nmoves, 0);
  // ensemble.py:128-129 then RandomState.choice(p=...): cdf = cumsum(p); cdf /= cdf[-1]
  s.cdf.resize(nmoves);
  double run = 0.0;
  for (size_t k = 0; k < nmoves; ++k) {
    run += s.moves[k].weight / tot;
    s.cdf[k] = run;
  }
  for (size_t k = 0; k < nmoves; ++k) s.cdf[k] /= run;
  return EB_OK;
}

// ensemble.py:406 -- one move per step for the whole ensemble
size_t choose_move(const eb_ctx* c, const Schedule& s, uint64_t step) {
  if (s.moves.size() == 1) return 0;
  const u32x4 w = draw_words(c->seed, step, 0, TAG_MOVE, 0);
  const double u = u53(w.x, w.y);
  size_t idx = 0;
  while (idx + 1 < s.cdf.size() && !(s.cdf[idx] > u)) ++idx;  // searchsorted(side="right")
  return idx;
}

void split_starts(int64_t N, int P, int* start) {
  start[0] = 0;
  for (int j = 0; j < P; ++j) start[j + 1] = start[j] + (int)((N - j + P - 1) / P);
}

void fill_base_args(eb_ctx* c, const eb_move& mv, HalfStepArgs& a) {
  a = HalfStepArgs{};
  a.coords = c->coords;
  a.logp = c->logp;
  a.accepted = c->accepted;
  a.nacc = c->nacc;
  a.status = c->status_dev;
  a.N = c->N;
  a.D = c->D;
  a.seed = c->seed;
  a.model = c->model;
  if (c->debug) {
    a.tap_partners = c->tap_partners;
    a.tap_scalar = c->tap_scalar;
    a.tap_u = c->tap_u;
    a.tap_active = c->tap_active;
  }
  switch (mv.kind) {
    case EB_MOVE_STRETCH:
      a.p0 = mv.p0;
      break;
    case EB_MOVE_DE:
      a.p0 = isnan(mv.p1) ? 2.38 / sqrt(2.0 * (double)c->D) : mv.p1;  // de.py:33-38
      a.p1 = mv.p0;                                                    // sigma
      break;
    default:
      a.p0 = mv.p0;  // gammas
  }
  a.timeline = c->timeline;
  a.dmma_stagger = c->dmma_stagger;
  comm_fill_args(c->comm, a);
}

bool dmma_eligible(const eb_ctx* c, const eb_move& mv) {
  return c->allow_dmma && mv.kind == EB_MOVE_STRETCH && c->model.kind == EB_MODEL_GAUSS_DENSE &&
         c->model.chol != nullptr && !c->debug;
}

int check_walker_count(eb_ctx* c, const eb_move& mv) {
  if (c->N < 2 * (int64_t)c->D && !mv.live_dangerously)  // red_blue.py:64-70
    FAIL(c, EB_ERR_FEW_WALKERS,
         "It is unadvisable to use a red-blue move with fewer walkers than twice the number of dimensions.");
  return EB_OK;
}

// launch the P half-steps of one step with the generic kernels (one launch per split)
int launch_step_generic(eb_ctx* c, const eb_move& mv, uint64_t step, const int32_t* order, size_t step_in_chunk,
                        uint64_t& launches) {
  const int P = mv.nsplits;
  int rc = check_walker_count(c, mv);
  if (rc) return rc;
  int start[MAX_SPLITS + 1];
  split_starts(c->N, P, start);
  HalfStepArgs a;
  fill_base_args(c, mv, a);
  a.order = order;
  a.step = step;
  for (int split = 0; split < P; ++split) {
    a.split = split;
    a.a_start = start[split];
    a.a_count = start[split + 1] - start[split];
    int k = 0;
    for (int j = 0; j < P && k < 3; ++j) {
      if (j == split) continue;
      a.c_start[k] = start[j];
      a.c_count[k] = start[j + 1] - start[j];
      ++k;
    }
    comm_active_range(c->comm, a, step_in_chunk);  // i_lo / i_hi for this rank
    if (c->fused_last) {
      // the previous launch was a dense_dmma kernel that carried the peer barrier itself (signal at its end);
      // this kernel does not wait on its own, so the ranks meet explicitly before it reads peer rows
      if (comm_barrier(c->comm, c->st, c->status_dev, launches)) FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
      c->fused_last = false;
    }
    c->chain_ok = false;
    bool used_tma = false;
    if (c->allow_tma && !c->debug)
      CK(c, launch_half_step_tma(mv.kind, a, capped_grid(c, c->sm_count), c->allow_tma >= 2, c->tma_own_reg, c->st,
                                 &used_tma, &c->last_shape));
    if (used_tma) {
      c->last_kernel = "tma_rows";
    } else {
      CK(c, launch_half_step_generic(mv.kind, a, c->st, &c->last_shape));
      c->last_kernel = "generic";
    }
    ++launches;
    c->tap_count = a.a_count;
    if (comm_after_split(c->comm, c->st, c->status_dev, launches)) FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
  }
  return EB_OK;
}

int ensure_move_scratch(eb_ctx* c) {
  const size_t D = (size_t)c->D;
  if (!c->qbuf) CK(c, cudaMalloc(&c->qbuf, (size_t)c->N * D * sizeof(double)));
  if (!c->walk_work && D <= 1024) CK(c, cudaMalloc(&c->walk_work, (2 * D + 3 * D * D) * sizeof(double)));
  if (!c->mom_partial && D <= 1024) CK(c, cudaMalloc(&c->mom_partial, moments_partial_bytes(c->D, c->sm_count)));
  return EB_OK;
}

// WalkMove (walk.py:27-37): per split a proposal kernel writes q[a_count, D], then the fused
// log-prob + accept + update kernel consumes it
int launch_step_walk(eb_ctx* c, const eb_move& mv, uint64_t step, const int32_t* order, uint64_t& launches) {
  const int P = mv.nsplits;
  int rc = check_walker_count(c, mv);
  if (rc) return rc;
  rc = ensure_move_scratch(c);
  if (rc) return rc;
  int start[MAX_SPLITS + 1];
  split_starts(c->N, P, start);
  HalfStepArgs a;
  fill_base_args(c, mv, a);
  a.order = order;
  a.step = step;
  a.qbuf = c->qbuf;
  c->chain_ok = false;
  const size_t D = (size_t)c->D;
  double* shift = c->walk_work;
  double* acc = shift + D;
  double* cov = acc + D + D * D;
  double* L = cov + D * D;
  for (int split = 0; split < P; ++split) {
    a.split = split;
    a.a_start = start[split];
    a.a_count = start[split + 1] - start[split];
    a.i_lo = 0;
    a.i_hi = a.a_count;
    a.range = nullptr;
    const int64_t Nc = c->N - a.a_count;
    const int64_t s0 = isnan(mv.p0) ? Nc : (int64_t)mv.p0;  // walk.py:32
    if (s0 == Nc) {
      // every walker of the split draws from the covariance of the WHOLE complement (walk.py:34-35 with a
      // permutation of all Nc rows): computed once -- moment sums on the tensor pipe, then a D x D factorisation
      CK(c, launch_colmean(c->coords, c->N, c->D, shift, nullptr, c->st));  // any shift will do: the ensemble mean
      CK(c, cudaMemsetAsync(acc, 0, (D + D * D) * sizeof(double), c->st));
      CK(c, launch_moments(c->coords, Nc, c->D, shift, c->mom_partial, acc, c->sm_count, c->st, order, a.a_start,
                           a.a_count));
      CK(c, launch_cov_chol(acc, (double)Nc, c->D, cov, L, c->st));
      CK(c, launch_walk_shared_propose(a, L, c->qbuf, c->st));
      launches += 5;
    } else {
      CK(c, launch_walk_subset_propose(a, (int)s0, c->qbuf, c->st));
      ++launches;
    }
    CK(c, launch_half_step_generic(MOVE_PRECOMPUTED, a, c->st));
    ++launches;
  }
  c->last_kernel = "walk";
  return EB_OK;
}

// MHMove with the Gaussian proposal (mh.py:35-65, gaussian.py:72-119): every walker is proposed at once
int launch_step_gaussian(eb_ctx* c, const Schedule& s, size_t mi, uint64_t step, uint64_t& launches) {
  const eb_move& mv = s.moves[mi];
  int rc = ensure_move_scratch(c);
  if (rc) return rc;
  const int D = c->D;
  double f = 1.0;
  if (!isnan(mv.p1)) {  // gaussian.py:88-91  exp(uniform(-log f, log f))
    const u32x4 w = draw_words(c->seed, step, 0, TAG_MOVE, 1);
    const double lf = log(mv.p1);
    f = exp(-lf + (lf - (-lf)) * u53(w.x, w.y));
  }
  const int seq_dim = (int)(((uint64_t)mv.seq_index + c->picks[mi]) % (uint64_t)D);  // gaussian.py:102-103
  const double* dev = c->gauss_dev + s.goff[mi];
  const int form = s.gform[mi];
  const double* scale = dev;
  c->chain_ok = false;
  if (form == 2) {
    double* v = c->gauss_dev + s.goff[mi] + (size_t)D * D;
    CK(c, launch_gaussian_shift(dev, D, f, c->seed, step, v, c->st));
    scale = v;
    ++launches;
  }
  CK(c, launch_gaussian_propose(c->coords, 0, c->N, D, form, scale, f, mv.mode, seq_dim, c->seed, step, c->qbuf, c->st));
  HalfStepArgs a;
  fill_base_args(c, mv, a);
  a.order = nullptr;  // the active set is every walker, in walker order
  a.step = step;
  a.split = 0;
  a.a_start = 0;
  a.a_count = (int)c->N;
  a.i_lo = 0;
  a.i_hi = (int)c->N;
  a.range = nullptr;
  a.qbuf = c->qbuf;
  CK(c, launch_half_step_generic(MOVE_PRECOMPUTED, a, c->st));
  launches += 2;
  c->last_kernel = "gaussian";
  return EB_OK;
}

constexpr int DMMA_TILE_SLOTS = 8;  // consumer warps per SM of the dense_dmma kernel

// a run of consecutive half-steps handed to ONE persistent dense_dmma launch
struct DmmaGroup {
  size_t first = 0;  // index into the chunk's HalfDesc array
  int nhalf = 0;
  int max_count = 0;
};

int flush_dmma(eb_ctx* c, const eb_move& mv, DmmaGroup& grp, uint64_t& launches) {
  if (grp.nhalf == 0) return EB_OK;
  HalfStepArgs a;
  fill_base_args(c, mv, a);
  a.order = c->order;  // chunk base; HalfDesc::order_step selects the table
  a.range = c->comm.nranks > 1 ? c->comm.ranges : nullptr;
  int bound = grp.max_count;
  if (c->comm.nranks > 1 && c->comm.rows_per_rank < bound) bound = (int)c->comm.rows_per_rank;
  // Locality-sorted tiles hide the peer barrier and the first remote fetch behind local work, but move the
  // remote burst to the second round: measured (profiles/r02_ab_2gpu.md) +4 % for strong scaling on 2 GPUs,
  // -4 % for weak scaling on 2 GPUs and -6 % for strong scaling on 4 GPUs -- hence off by default; "auto"
  // (option value 1) enables it when a consumer warp has at most ~2 tiles per half-step.
  const bool few_tiles = (bound + 7) / 8 <= 2 * DMMA_TILE_SLOTS * c->sm_count;
  a.aperm = (c->comm.nranks > 1 && (c->local_first == 2 || (c->local_first == 1 && few_tiles))) ? c->comm.aperm : nullptr;
  // P2P: the peer barrier rides inside the kernel (wait at its start, between its half-steps, signal at its end)
  const bool fused = comm_fuse_barrier(c->comm, a, grp.nhalf);
  c->fused_last = fused;
  // (sharded ensembles: measured slower with the dependent launch -- the early CTAs only add pollers on the
  // peer flags -- so it is opt-in there: option "pdl" = 2)
  const bool pdl = c->chain_ok && grp.nhalf == 1 && (c->comm.nranks > 1 ? c->pdl >= 2 : c->pdl >= 1);
  CK(c, launch_dense_dmma(a, c->descs_host[grp.first], c->descs_dev + grp.first, grp.nhalf, bound, c->gbar, c->gbar_count,
                          capped_grid(c, c->sm_count), pdl, &c->last_shape, c->st));
  const int grid = (int)c->last_shape.grid;
  c->gbar_count += (unsigned long long)(grp.nhalf - 1) * (unsigned long long)grid;
  c->last_kernel = "dense_dmma";
  c->chain_ok = grid > 0;
  ++launches;
  grp = DmmaGroup{};
  return EB_OK;
}

// run nsteps steps.  `after_step(k)` is called with the work of step k enqueued and may
// enqueue copies on the stream; `sync_every` > 0 tells how often it actually does (every
// sync_every-th step), so that steps in between can share one persistent launch.
int accumulate_moments(eb_ctx* c, uint64_t& launches);  // below

template <class F>
int run_steps(eb_ctx* c, const Schedule& s, uint64_t nsteps, uint64_t sync_every, F&& after_step) {
  uint64_t launches = 0;
  const bool perstep = c->l2_flush;  // flush L2 before every step, time each step on its own
  if (perstep) {
    if (nsteps > 16384) FAIL(c, EB_ERR_INVALID, "l2_flush mode times each step separately; use nsteps <= 16384");
    if (!c->flush_buf) CK(c, cudaMalloc(&c->flush_buf, c->flush_bytes));
    while (c->ev_pool.size() < 2 * nsteps) {
      cudaEvent_t e;
      CK(c, cudaEventCreate(&e));
      c->ev_pool.push_back(e);
    }
  }
  c->chain_ok = false;
  CK(c, cudaEventRecord(c->ev0, c->st));
  if (comm_begin(c->comm, c->st, c->status_dev, launches)) FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
  c->fused_last = false;
  const bool multi = c->comm.nranks > 1;
  // sharded ensembles run one half-step per launch: NCCL exchanges whole row blocks after every split, and the
  // P2P peer barrier rides on the kernel boundary (a persistent launch with the peer barrier between its
  // half-steps measured no faster -- profiles/r02_ab_2gpu.md -- and was dropped)
  const bool one_per_launch = multi;
  const bool exchange_each = multi && c->comm.mode == EB_COMM_ALLGATHER;
  std::vector<size_t> pick;
  uint64_t done = 0;
  while (done < nsteps) {
    const size_t chunk = (size_t)std::min<uint64_t>(nsteps - done, c->table_cap);
    pick.resize(chunk);
    CK(c, cudaStreamSynchronize(c->st));  // info_host / descs_host are reused per chunk
    size_t ndesc = 0;
    for (size_t k = 0; k < chunk; ++k) {
      pick[k] = choose_move(c, s, c->step + k);
      const eb_move& mv = s.moves[pick[k]];
      c->info_host[k].nsplits = mv.nsplits;
      c->info_host[k].randomize = mv.randomize_split;
    }
    // Split tables depend only on (seed, step, nsplits, randomize): reuse the ones already on the
    // device when they cover this chunk, else build them -- looking ahead with the same schedule, so
    // a caller that steps one iteration per call pays for one table launch every 64 calls, not one each.
    size_t off = 0, build = 0;
    bool hit = c->tbl_n > 0 && c->tbl_seed == c->seed && c->step >= c->tbl_step0 &&
               c->step + chunk <= c->tbl_step0 + c->tbl_n;
    if (hit) {
      off = (size_t)(c->step - c->tbl_step0);
      for (size_t k = 0; k < chunk && hit; ++k)
        hit = c->tbl_info[off + k].nsplits == c->info_host[k].nsplits &&
              c->tbl_info[off + k].randomize == c->info_host[k].randomize;
    }
    if (!hit) {
      off = 0;
      build = std::min<size_t>(c->table_cap, std::max<size_t>(chunk, 64));
      for (size_t k = chunk; k < build; ++k) {
        const eb_move& mv = s.moves[choose_move(c, s, c->step + k)];
        c->info_host[k].nsplits = mv.nsplits;
        c->info_host[k].randomize = mv.randomize_split;
      }
      c->tbl_seed = c->seed;
      c->tbl_step0 = c->step;
      c->tbl_n = build;
      c->tbl_info.assign(c->info_host, c->info_host + build);
    }
    for (size_t k = 0; k < chunk; ++k) {
      const eb_move& mv = s.moves[pick[k]];
      if (dmma_eligible(c, mv)) {
        int start[MAX_SPLITS + 1];
        split_starts(c->N, mv.nsplits, start);
        for (int split = 0; split < mv.nsplits; ++split) {
          HalfDesc& d = c->descs_host[ndesc++];
          d.step = c->step + k;
          d.order_step = (int32_t)(off + k);
          d.split = split;
          d.a_start = start[split];
          d.a_count = start[split + 1] - start[split];
        }
      }
    }
    DmmaGroup grp;
    size_t desc_cursor = 0;
    const eb_move* grp_move = nullptr;
    for (size_t k = 0; k < chunk; ++k) {
      const eb_move& mv = s.moves[pick[k]];
      if (perstep) {
        CK(c, cudaMemsetAsync(c->flush_buf, (int)(k & 0xff), c->flush_bytes, c->st));
        CK(c, cudaEventRecord(c->ev_pool[2 * (done + k)], c->st));
        c->chain_ok = false;
      }
      if (k == 0) {
        // dense_dmma descriptors of the chunk and, when needed, the split tables (charged to this step)
        if (ndesc) {
          CK(c, cudaMemcpyAsync(c->descs_dev, c->descs_host, ndesc * sizeof(HalfDesc), cudaMemcpyHostToDevice, c->st));
          c->chain_ok = false;
        }
        if (build) {
          CK(c, cudaMemcpyAsync(c->info_dev, c->info_host, build * sizeof(StepInfo), cudaMemcpyHostToDevice, c->st));
          const Comm& cm = c->comm;
          CK(c, launch_split_tables(c->order, c->info_dev, (int)build, c->N, c->seed, c->step,
                                    cm.rows_per_rank * cm.rank, cm.rows_per_rank * (cm.rank + 1),
                                    cm.nranks > 1 ? cm.ranges : nullptr, c->st));
          ++launches;
          if (cm.nranks > 1 && cm.aperm) {
            // front group = one tile (8 walkers) for each of the 8 consumer warps of every SM: the first round
            CK(c, launch_locality_tables(c->order, c->info_dev, cm.ranges, (int)build, c->N, c->seed, c->step,
                                         cm.rows_per_rank, cm.rank, 64 * c->sm_count, cm.aperm, c->st));
            ++launches;
          }
          c->chain_ok = false;
        }
      }
      int rc;
      if (dmma_eligible(c, mv)) {
        rc = check_walker_count(c, mv);
        if (rc) return rc;
        if (grp_move && grp_move != &mv) {  // a different move object: its parameters differ
          rc = flush_dmma(c, *grp_move, grp, launches);
          if (rc) return rc;
        }
        grp_move = &mv;
        for (int split = 0; split < mv.nsplits; ++split) {
          const HalfDesc& d = c->descs_host[desc_cursor];
          if (grp.nhalf == 0) grp.first = desc_cursor;
          grp.nhalf += 1;
          grp.max_count = std::max(grp.max_count, (int)d.a_count);
          ++desc_cursor;
          if (one_per_launch || (grp.nhalf >= c->dmma_group && split + 1 < mv.nsplits)) {
            rc = flush_dmma(c, mv, grp, launches);
            if (rc) return rc;
            if (exchange_each) {
              c->chain_ok = false;
              if (comm_after_split(c->comm, c->st, c->status_dev, launches))
                FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
            }
          }
        }
        const bool moments_now = c->moments_every > 0 && (c->step + 1) % c->moments_every == 0;
        const bool host_event = perstep || moments_now || (sync_every > 0 && (done + k + 1) % sync_every == 0);
        if (host_event || k + 1 == chunk || grp.nhalf >= c->dmma_group) {
          rc = flush_dmma(c, mv, grp, launches);
          if (rc) return rc;
        }
      } else {
        if (grp_move) {
          rc = flush_dmma(c, *grp_move, grp, launches);
          if (rc) return rc;
        }
        if (mv.kind == EB_MOVE_WALK)
          rc = launch_step_walk(c, mv, c->step, c->order + (off + k) * (size_t)c->N, launches);
        else if (mv.kind == EB_MOVE_GAUSSIAN)
          rc = launch_step_gaussian(c, s, pick[k], c->step, launches);
        else
          rc = launch_step_generic(c, mv, c->step, c->order + (off + k) * (size_t)c->N, off + k, launches);
        if (rc) return rc;
      }
      c->picks[pick[k]] += 1;
      c->step += 1;
      if (c->moments_every > 0 && c->step % c->moments_every == 0) {
        rc = accumulate_moments(c, launches);
        if (rc) return rc;
      }
      if (perstep) {
        CK(c, cudaEventRecord(c->ev_pool[2 * (done + k) + 1], c->st));
        c->chain_ok = false;
      }
      rc = after_step(done + k);
      if (rc) return rc;
    }
    done += chunk;
  }
  CK(c, cudaEventRecord(c->ev1, c->st));
  c->chain_ok = false;
  // multi-GPU: the rows of other ranks are NOT replicated here; collective readers (eb_get_state,
  // eb_get_naccepted, the accept mask of eb_step) do that on demand, sharded readers never need it
  if (multi) c->replicas_dirty = true;
  CK(c, cudaMemcpyAsync(c->status_host, c->status_dev, sizeof(int), cudaMemcpyDeviceToHost, c->st));
  CK(c, cudaStreamSynchronize(c->st));
  float ms = 0.f;
  if (perstep) {
    double tot = 0.0;
    for (uint64_t k = 0; k < nsteps; ++k) {
      CK(c, cudaEventElapsedTime(&ms, c->ev_pool[2 * k], c->ev_pool[2 * k + 1]));
      tot += ms;
    }
    c->last_ms = tot;
  } else {
    CK(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    c->last_ms = ms;
  }
  c->last_launches = launches;
  return check_status(c);
}

// ---- running chain moments ---------------------------------------------------------------------
int moments_config(eb_ctx* c, uint64_t every) {
  CK(c, cudaSetDevice(c->device));
  if (every > 0 && c->D > 1024) FAIL(c, EB_ERR_UNSUPPORTED, "chain moments are limited to ndim <= 1024");
  const size_t n = (size_t)c->D + (size_t)c->D * c->D;
  if (every > 0 && !c->mom_acc) {
    CK(c, cudaMalloc(&c->mom_acc, n * sizeof(double)));
    CK(c, cudaMalloc(&c->mom_shift, (size_t)c->D * sizeof(double)));
    if (!c->mom_partial) CK(c, cudaMalloc(&c->mom_partial, moments_partial_bytes(c->D, c->sm_count)));
  }
  if (c->mom_acc) CK(c, cudaMemsetAsync(c->mom_acc, 0, n * sizeof(double), c->st));
  c->mom_count = 0;
  c->mom_have_shift = false;
  c->moments_every = every;
  CK(c, cudaStreamSynchronize(c->st));
  return EB_OK;
}

// fold the rows this rank owns of the CURRENT state into the accumulators (enqueued on the stream)
int accumulate_moments(eb_ctx* c, uint64_t& launches) {
  int64_t r0, r1;
  owned_rows(c, r0, r1);
  const double* X = c->coords + (size_t)r0 * c->D;
  c->chain_ok = false;
  if (!c->mom_have_shift) {
    // shift = the ensemble mean at the first accumulation: keeps the raw second moments well conditioned
    CK(c, launch_colmean(X, r1 - r0, c->D, c->mom_shift, nullptr, c->st));
    c->mom_have_shift = true;
    ++launches;
  }
  CK(c, launch_moments(X, r1 - r0, c->D, c->mom_shift, c->mom_partial, c->mom_acc, c->sm_count, c->st));
  launches += 2;
  c->mom_count += (unsigned long long)(r1 - r0);
  return EB_OK;
}

int step_preflight(eb_ctx* c) {
  if (!c->have_model) FAIL(c, EB_ERR_STATE, "eb_step: no model set");
  if (!c->have_state) FAIL(c, EB_ERR_STATE, "eb_step: no state set");
  CK(c, cudaSetDevice(c->device));
  return EB_OK;
}

}  // namespace

extern "C" {

int eb_step(eb_ctx* c, const eb_move* moves, size_t nmoves, uint64_t nsteps, uint8_t* accepted_last) {
  if (!c) return EB_ERR_INVALID;
  int rc = step_preflight(c);
  if (rc) return rc;
  Schedule s;
  rc = build_schedule(c, moves, nmoves, s);
  if (rc) return rc;
  if (nsteps > 0) {
    rc = run_steps(c, s, nsteps, 0, [](uint64_t) { return EB_OK; });
    if (rc) return rc;
  }
  if (accepted_last) {
    rc = sync_replicas(c);  // multi-GPU: the mask of every rank's rows (collective)
    if (rc) return rc;
    CK(c, cudaMemcpyAsync(accepted_last, c->accepted, (size_t)c->N, cudaMemcpyDeviceToHost, c->st));
    CK(c, cudaStreamSynchronize(c->st));
  }
  return EB_OK;
}

int eb_step_store(eb_ctx* c, const eb_move* moves, size_t nmoves, uint64_t nsteps, uint64_t thin_by,
                  double* chain, double* log_prob, double* accepted) {
  if (!c) return EB_ERR_INVALID;
  if (thin_by == 0) FAIL(c, EB_ERR_INVALID, "Invalid thinning argument");  // ensemble.py:380-381
  if (!chain || !log_prob) FAIL(c, EB_ERR_INVALID, "eb_step_store: null output buffer");
  int rc = step_preflight(c);
  if (rc) return rc;
  Schedule s;
  rc = build_schedule(c, moves, nmoves, s);
  if (rc) return rc;
  const size_t N = (size_t)c->N, D = (size_t)c->D;
  const size_t row = N * D + N;  // coords then log_prob, staged together
  for (int k = 0; k < 2; ++k) {
    if (!c->stage[k]) {
      CK(c, cudaMallocHost(&c->stage[k], row * sizeof(double)));
      CK(c, cudaMallocHost(&c->stage_acc[k], N));
      CK(c, cudaEventCreateWithFlags(&c->stage_ev[k], cudaEventDisableTiming));
    }
  }
  // double-buffered pinned staging: the D2H of stored step k overlaps the
  // kernels of the following steps; the host drains slot k-1 while k is in flight
  uint64_t stored = 0;
  int64_t pending[2] = {-1, -1};
  auto drain = [&](int slot) -> int {
    if (pending[slot] < 0) return EB_OK;
    CK(c, cudaEventSynchronize(c->stage_ev[slot]));
    const size_t k = (size_t)pending[slot];
    memcpy(chain + k * N * D, c->stage[slot], N * D * sizeof(double));          // backend.py:224
    memcpy(log_prob + k * N, c->stage[slot] + N * D, N * sizeof(double));        // backend.py:225
    if (accepted)
      for (size_t w = 0; w < N; ++w) accepted[w] += (double)c->stage_acc[slot][w];  // backend.py:229
    pending[slot] = -1;
    return EB_OK;
  };
  rc = run_steps(c, s, nsteps, thin_by, [&](uint64_t k) -> int {
    if ((k + 1) % thin_by != 0) return EB_OK;  // ensemble.py:416
    const int slot = (int)(stored & 1);
    int r = drain(slot);
    if (r) return r;
    c->chain_ok = false;
    if (c->comm.nranks > 1) {
      // a stored step holds EVERY walker: replicate the other ranks' rows (log_prob, accept mask and, in
      // P2P mode, coords) before the copy -- the in-run exchange only moves what the kernels need
      uint64_t l = 0;
      if (comm_sync_state(c->comm, c->st, c->status_dev, c->logp, c->accepted, nullptr, l))
        FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
      c->fused_last = false;
    }
    CK(c, cudaMemcpyAsync(c->stage[slot], c->coords, N * D * sizeof(double), cudaMemcpyDeviceToHost, c->st));
    CK(c, cudaMemcpyAsync(c->stage[slot] + N * D, c->logp, N * sizeof(double), cudaMemcpyDeviceToHost, c->st));
    CK(c, cudaMemcpyAsync(c->stage_acc[slot], c->accepted, N, cudaMemcpyDeviceToHost, c->st));
    CK(c, cudaEventRecord(c->stage_ev[slot], c->st));
    pending[slot] = (int64_t)stored;
    ++stored;
    return EB_OK;
  });
  int r0 = drain((int)(stored & 1));
  int r1 = drain((int)((stored + 1) & 1));
  if (rc) return rc;
  if (r0) return r0;
  return r1;
}

int eb_get_naccepted(eb_ctx* c, uint64_t* naccepted) {
  if (!c || !naccepted) return EB_ERR_INVALID;
  CK(c, cudaSetDevice(c->device));
  int rc = sync_replicas(c);  // multi-GPU: every rank's counters (collective)
  if (rc) return rc;
  CK(c, cudaMemcpyAsync(naccepted, c->nacc, (size_t)c->N * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->st));
  CK(c, cudaStreamSynchronize(c->st));
  return EB_OK;
}

int eb_move_picks(const eb_ctx* c, uint64_t* picks, size_t nmoves) {
  if (!c || !picks) return EB_ERR_INVALID;
  for (size_t k = 0; k < nmoves; ++k) picks[k] = k < c->picks.size() ? c->picks[k] : 0;
  return EB_OK;
}

int eb_reset_counters(eb_ctx* c) {
  if (!c) return EB_ERR_INVALID;
  CK(c, cudaSetDevice(c->device));
  CK(c, cudaMemsetAsync(c->nacc, 0, (size_t)c->N * sizeof(unsigned long long), c->st));
  CK(c, cudaStreamSynchronize(c->st));
  return EB_OK;
}

int eb_moments(eb_ctx* c, double* mean, double* cov, uint64_t* count, uint64_t* naccepted_total) {
  if (!c) return EB_ERR_INVALID;
  if (!c->mom_acc) FAIL(c, EB_ERR_STATE, "eb_moments: enable with eb_set_option(\"moments_every\", n) before stepping");
  CK(c, cudaSetDevice(c->device));
  const size_t D = (size_t)c->D, n = D + D * D;
  std::vector<double> acc(n), shift(D);
  CK(c, cudaMemcpyAsync(acc.data(), c->mom_acc, n * sizeof(double), cudaMemcpyDeviceToHost, c->st));
  CK(c, cudaMemcpyAsync(shift.data(), c->mom_shift, D * sizeof(double), cudaMemcpyDeviceToHost, c->st));
  std::vector<unsigned long long> nacc;
  int64_t r0, r1;
  owned_rows(c, r0, r1);
  if (naccepted_total) {
    nacc.resize((size_t)(r1 - r0));
    CK(c, cudaMemcpyAsync(nacc.data(), c->nacc + r0, nacc.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                          c->st));
  }
  CK(c, cudaStreamSynchronize(c->st));
  c->chain_ok = false;
  const double m = (double)c->mom_count;
  if (count) *count = c->mom_count;
  if (naccepted_total) {
    unsigned long long tot = 0;
    for (unsigned long long v : nacc) tot += v;
    *naccepted_total = tot;
  }
  if (c->mom_count == 0) {
    if (mean) std::fill(mean, mean + D, NAN);
    if (cov) std::fill(cov, cov + D * D, NAN);
    return EB_OK;
  }
  // mean = shift + S1 / m ; cov = (S2 - S1 S1^T / m) / (m - 1)   (np.cov(flatchain, rowvar=False))
  if (mean)
    for (size_t d = 0; d < D; ++d) mean[d] = shift[d] + acc[d] / m;
  if (cov)
    for (size_t r = 0; r < D; ++r)
      for (size_t k = 0; k < D; ++k)
        cov[r * D + k] = (acc[D + r * D + k] - acc[r] * acc[k] / m) / (m - 1.0);
  return EB_OK;
}

int eb_walkers_gram(eb_ctx* c, const double* coords, size_t rows, double* gram, int* flags) {
  if (!c) return EB_ERR_INVALID;
  if (!coords || !gram || rows == 0) FAIL(c, EB_ERR_INVALID, "eb_walkers_gram: null buffer");
  if (c->D > 1024) FAIL(c, EB_ERR_UNSUPPORTED, "eb_walkers_gram is limited to ndim <= 1024");
  CK(c, cudaSetDevice(c->device));
  int rc = ensure_scratch(c, rows);
  if (rc) return rc;
  const size_t D = (size_t)c->D, n = D + D * D;
  double* work = nullptr;  // [D mean | D + D*D accumulators]
  CK(c, cudaMalloc(&work, (D + n) * sizeof(double)));
  if (!c->mom_partial) {
    cudaError_t e = cudaMalloc(&c->mom_partial, moments_partial_bytes(c->D, c->sm_count));
    if (e != cudaSuccess) {
      cudaFree(work);
      CK(c, e);
    }
  }
  c->chain_ok = false;
  std::vector<double> acc(n);
  int f = 0;
  cudaError_t e = cudaMemcpyAsync(c->scratch_x, coords, rows * D * sizeof(double), cudaMemcpyHostToDevice, c->st);
  if (e == cudaSuccess) e = cudaMemsetAsync(work, 0, (D + n) * sizeof(double), c->st);
  if (e == cudaSuccess) e = launch_colmean(c->scratch_x, (int64_t)rows, c->D, work, c->status_dev, c->st);
  if (e == cudaSuccess)
    e = launch_moments(c->scratch_x, (int64_t)rows, c->D, work, c->mom_partial, work + D, c->sm_count, c->st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(acc.data(), work + D, n * sizeof(double), cudaMemcpyDeviceToHost, c->st);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(c->status_host, c->status_dev, sizeof(int), cudaMemcpyDeviceToHost, c->st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->st);
  cudaFree(work);
  CK(c, e);
  // the non-finite flags are an ANSWER here (walkers_independent returns False), not an error
  if (*c->status_host & (FLAG_INF_PARAM | FLAG_NAN_PARAM)) f |= 1;
  *c->status_host = 0;
  CK(c, cudaMemsetAsync(c->status_dev, 0, sizeof(int), c->st));
  CK(c, cudaStreamSynchronize(c->st));
  // centred, column-normalised walkers C (ensemble.py:656-661): C^T C = M_jk / sqrt(M_jj M_kk); the
  // max-abs scaling of :658-659 cancels, it only matters as the zero-span test
  for (size_t j = 0; j < D; ++j)
    if (!(acc[D + j * D + j] > 0.0)) f |= 2;
  for (size_t j = 0; j < D; ++j)
    for (size_t k = 0; k < D; ++k) {
      const double den = sqrt(acc[D + j * D + j] * acc[D + k * D + k]);
      gram[j * D + k] = den > 0.0 ? acc[D + j * D + k] / den : 0.0;
    }
  if (flags) *flags = f;
  return EB_OK;
}

int eb_autocorr(eb_ctx* c, const double* chain, size_t n_t, size_t nw, size_t nd, double* acf) {
  if (!c) return EB_ERR_INVALID;
  if (!chain || !acf || n_t == 0 || nw == 0 || nd == 0) FAIL(c, EB_ERR_INVALID, "eb_autocorr: empty chain or null buffer");
  if (n_t > ((size_t)1 << 26) || nw * nd > ((size_t)1 << 31))
    FAIL(c, EB_ERR_UNSUPPORTED, "eb_autocorr: chain too long (n_step <= 2^26)");
  CK(c, cudaSetDevice(c->device));
  const int M = acf_fft_length(n_t);
  // slab of walkers sized to ~1 GiB of scratch (at least one walker)
  const size_t per_walker = acf_bytes_per_series(n_t) * nd;
  size_t wb = ((size_t)1 << 30) / per_walker;
  wb = std::max<size_t>(1, std::min(wb, nw));
  const size_t S = wb * nd;
  double *xin = nullptr, *mean = nullptr, *f = nullptr;
  double2 *z = nullptr, *tw = nullptr;
  auto release = [&]() {
    cudaFree(xin);
    cudaFree(mean);
    cudaFree(f);
    cudaFree(z);
    cudaFree(tw);
  };
#define AC(call)                                                                             \
  do {                                                                                       \
    cudaError_t _e = (call);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      cudaGetLastError();                                                                    \
      release();                                                                             \
      FAIL(c, EB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
    }                                                                                        \
  } while (0)
  AC(cudaMalloc(&xin, n_t * S * sizeof(double)));
  AC(cudaMalloc(&mean, S * sizeof(double)));
  AC(cudaMalloc(&f, nd * n_t * sizeof(double)));
  AC(cudaMalloc(&z, S * (size_t)M * sizeof(double2)));
  AC(cudaMalloc(&tw, (size_t)std::max(1, M / 2) * sizeof(double2)));
  c->chain_ok = false;
  AC(cudaMemsetAsync(f, 0, nd * n_t * sizeof(double), c->st));
  AC(launch_acf_twiddles(tw, M, c->st));
  for (size_t w0 = 0; w0 < nw; w0 += wb) {
    const size_t wn = std::min(wb, nw - w0);
    // chain[t][w0 .. w0 + wn)[:] -> xin[t][wn * nd]: one strided copy (rows of the slab are contiguous in a step)
    AC(cudaMemcpy2DAsync(xin, wn * nd * sizeof(double), chain + w0 * nd, nw * nd * sizeof(double),
                         wn * nd * sizeof(double), n_t, cudaMemcpyHostToDevice, c->st));
    AC(launch_acf_slab(xin, (int)n_t, (int)wn, (int)nd, M, tw, z, mean, f, c->st));
  }
  AC(launch_acf_scale(f, nd * n_t, 1.0 / (double)nw, c->st));  // autocorr.py:106  f /= n_w
  AC(cudaMemcpyAsync(acf, f, nd * n_t * sizeof(double), cudaMemcpyDeviceToHost, c->st));
  AC(cudaStreamSynchronize(c->st));
#undef AC
  release();
  return EB_OK;
}

int eb_last_step_timing(const eb_ctx* c, double* ms, uint64_t* launches) {
  if (!c) return EB_ERR_INVALID;
  if (ms) *ms = c->last_ms;
  if (launches) *launches = c->last_launches;
  return EB_OK;
}

const char* eb_last_kernel_name(const eb_ctx* c) { return c ? c->last_kernel : "none"; }

int eb_set_option(eb_ctx* c, const char* name, int64_t value) {
  if (!c || !name) return EB_ERR_INVALID;
  if (!strcmp(name, "debug_taps")) {
    CK(c, cudaSetDevice(c->device));
    if (value && !c->tap_scalar) {
      const size_t N = (size_t)c->N;
      CK(c, cudaMalloc(&c->tap_partners, 3 * N * sizeof(int64_t)));
      CK(c, cudaMalloc(&c->tap_scalar, N * sizeof(double)));
      CK(c, cudaMalloc(&c->tap_u, N * sizeof(double)));
      CK(c, cudaMalloc(&c->tap_active, N * sizeof(int64_t)));
    }
    c->debug = value != 0;
    return EB_OK;
  }
  if (!strcmp(name, "dmma_timeline")) {
    CK(c, cudaSetDevice(c->device));
    const size_t n = (size_t)c->sm_count * 8 * TL_TILES * TL_EVENTS;
    if (value && !c->timeline) {
      CK(c, cudaMalloc(&c->timeline, n * sizeof(long long)));
      CK(c, cudaMemset(c->timeline, 0, n * sizeof(long long)));
    } else if (!value && c->timeline) {
      cudaFree(c->timeline);
      c->timeline = nullptr;
    }
    return EB_OK;
  }
  if (!strcmp(name, "l2_flush")) {
    c->l2_flush = value != 0;
    return EB_OK;
  }
  if (!strcmp(name, "dmma_stagger")) {
    c->dmma_stagger = value != 0;
    return EB_OK;
  }
  if (!strcmp(name, "dmma_group")) {
    if (value < 1) FAIL(c, EB_ERR_INVALID, "dmma_group must be >= 1");
    c->dmma_group = (int)std::min<int64_t>(value, 1 << 20);
    return EB_OK;
  }
  if (!strcmp(name, "tma_own_reg")) {
    c->tma_own_reg = value != 0;
    return EB_OK;
  }
  if (!strcmp(name, "dmma_local_first")) {
    c->local_first = (int)std::max<int64_t>(0, std::min<int64_t>(value, 2));
    return EB_OK;
  }
  if (!strcmp(name, "pdl")) {
    c->pdl = (int)std::max<int64_t>(0, std::min<int64_t>(value, 2));
    return EB_OK;
  }
  if (!strcmp(name, "moments_every")) {
    if (value < 0) FAIL(c, EB_ERR_INVALID, "moments_every must be >= 0");
    return moments_config(c, (uint64_t)value);
  }
  if (!strcmp(name, "tma_rows")) {
    c->allow_tma = (int)std::max<int64_t>(0, std::min<int64_t>(value, 2));
    return EB_OK;
  }
  if (!strcmp(name, "dense_dmma")) {
    c->allow_dmma = value != 0;
    return EB_OK;
  }
  if (!strcmp(name, "grid_cap")) {
    if (value < 0) FAIL(c, EB_ERR_INVALID, "grid_cap must be >= 0");
    c->grid_cap = (int)std::min<int64_t>(value, 1 << 30);
    return EB_OK;
  }
  FAIL(c, EB_ERR_INVALID, "eb_set_option: unknown option '%s'", name);
}

int eb_debug_timeline(eb_ctx* c, int64_t* out, size_t capacity, size_t* written) {
  if (!c || !out) return EB_ERR_INVALID;
  if (!c->timeline) FAIL(c, EB_ERR_STATE, "eb_debug_timeline: enable with eb_set_option(\"dmma_timeline\", 1)");
  CK(c, cudaSetDevice(c->device));
  const size_t n = (size_t)c->sm_count * 8 * TL_TILES * TL_EVENTS;
  if (capacity < n) FAIL(c, EB_ERR_INVALID, "eb_debug_timeline: need room for %zu values", n);
  CK(c, cudaMemcpy(out, c->timeline, n * sizeof(long long), cudaMemcpyDeviceToHost));
  if (written) *written = n;
  return EB_OK;
}

int eb_debug_taps(eb_ctx* c, int64_t* partners, double* scalar, double* u_accept, int64_t* active,
                  int64_t* nactive) {
  if (!c) return EB_ERR_INVALID;
  if (!c->debug || !c->tap_scalar) FAIL(c, EB_ERR_STATE, "eb_debug_taps: enable with eb_set_option(\"debug_taps\", 1)");
  CK(c, cudaSetDevice(c->device));
  const size_t N = (size_t)c->N;
  if (partners) CK(c, cudaMemcpy(partners, c->tap_partners, 3 * N * sizeof(int64_t), cudaMemcpyDeviceToHost));
  if (scalar) CK(c, cudaMemcpy(scalar, c->tap_scalar, N * sizeof(double), cudaMemcpyDeviceToHost));
  if (u_accept) CK(c, cudaMemcpy(u_accept, c->tap_u, N * sizeof(double), cudaMemcpyDeviceToHost));
  if (active) CK(c, cudaMemcpy(active, c->tap_active, N * sizeof(int64_t), cudaMemcpyDeviceToHost));
  if (nactive) *nactive = c->tap_count;
  return EB_OK;
}

int eb_debug_launch_config(const eb_ctx* c, int64_t* out, size_t n) {
  if (!c || !out || n < EB_LAUNCH_CONFIG_FIELDS) return EB_ERR_INVALID;
  static_assert(sizeof(LaunchShape) == EB_LAUNCH_CONFIG_FIELDS * sizeof(int64_t), "one int64 per field");
  memcpy(out, &c->last_shape, sizeof(LaunchShape));
  return EB_OK;
}

int eb_host_alloc(size_t bytes, void** out) {
  if (!out || bytes == 0) return EB_ERR_INVALID;
  if (cudaMallocHost(out, bytes) != cudaSuccess) {
    cudaGetLastError();
    *out = nullptr;
    return EB_ERR_CUDA;
  }
  return EB_OK;
}

int eb_host_free(void* ptr) {
  if (ptr && cudaFreeHost(ptr) != cudaSuccess) {
    cudaGetLastError();
    return EB_ERR_CUDA;
  }
  return EB_OK;
}

// ---- multi-GPU ---------------------------------------------------------------
int eb_comm_id(char id[EB_COMM_ID_BYTES]) { return comm_unique_id(id) ? EB_ERR_COMM : EB_OK; }

int eb_comm_init(eb_ctx* c, const char id[EB_COMM_ID_BYTES], int rank, int nranks, int mode) {
  if (!c) return EB_ERR_INVALID;
  CK(c, cudaSetDevice(c->device));
  c->tbl_n = 0;  // the cached split tables carry the old ownership ranges
  c->have_state = false;  // ownership changes: the state must be set again through the sharded path
  unsigned* flags = reinterpret_cast<unsigned*>(c->coords + (size_t)c->N * c->D);
  if (comm_init(c->comm, id, rank, nranks, mode, c->N, c->D, c->coords, flags, c->table_cap, c->st))
    FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
  return EB_OK;
}

int eb_comm_export(eb_ctx* c, char blob[EB_IPC_BLOB_BYTES]) {
  if (!c) return EB_ERR_INVALID;
  CK(c, cudaSetDevice(c->device));
  if (comm_export(c->comm, blob)) FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
  return EB_OK;
}

int eb_comm_probe(eb_ctx* c, int peer, int what, double* gbs) {
  if (!c || !gbs) return EB_ERR_INVALID;
  CK(c, cudaSetDevice(c->device));
  if (comm_probe(c->comm, peer, what, c->D, c->st, gbs)) FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
  return EB_OK;
}

int eb_comm_import(eb_ctx* c, const char* blobs) {
  if (!c) return EB_ERR_INVALID;
  CK(c, cudaSetDevice(c->device));
  if (comm_import(c->comm, blobs)) FAIL(c, EB_ERR_COMM, "%s", c->comm.err.c_str());
  return EB_OK;
}

}  // extern "C"
