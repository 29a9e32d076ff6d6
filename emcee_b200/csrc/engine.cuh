// Internal types shared by the kernels and the C ABI (not part of the boundary).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/emcee_b200.h"
#include "philox.cuh"

namespace eb {

constexpr int MAX_SPLITS = 32;      // split_table_kernel uses one warp per set
constexpr int TABLE_THREADS = 1024;
constexpr int TL_TILES = 8, TL_EVENTS = 10;  // dense_dmma timeline buffer shape (6 consumer + 4 producer stamps)

// device status flags (OR-ed by kernels, read back after every call)
enum : int {
  FLAG_NAN_LOGPROB = 1,
  FLAG_INF_PARAM = 2,
  FLAG_NAN_PARAM = 4,
  FLAG_COMM_TIMEOUT = 8,
};

struct ModelDev {
  int kind;
  const double* params;  // device: gauss_dense mu[D], A[D*D]; else unused
  const double* chol;    // device: gauss_dense packed factor for the DMMA kernel (or null)
  double s0, s1;         // rosenbrock a,b ; ring R,sigma
};

// per-step split description handed to split_table_kernel
struct StepInfo {
  int32_t nsplits;
  int32_t randomize;
};

// everything one half-step (one split of one step) needs
struct HalfStepArgs {
  double* coords;            // [N, D] row-major, live state
  double* logp;              // [N]
  uint8_t* accepted;         // [N] accept mask of the current step
  unsigned long long* nacc;  // [N] accepted-proposal counters
  int* status;               // flags
  const int32_t* order;      // [N] walker ids grouped by set, ascending inside a set
  const double* const* peer_coords;  // P2P mode: [nranks] peer-mapped coords (or null)
  int64_t rows_per_rank;     // P2P mode: owner(w) = w / rows_per_rank
  // P2P mode, barrier fused into the kernel (dense_dmma): producers wait until every peer has
  // published p2p_wait before touching the state; the last CTA to finish publishes p2p_signal
  unsigned* const* p2p_peer_flags;  // [nranks] peer-mapped flag arrays (null: no fused barrier)
  const unsigned* p2p_my_flags;     // [nranks] this rank's flag array (written by the peers)
  unsigned* p2p_done;               // CTA-completion counter of this rank
  int p2p_rank, p2p_nranks;
  unsigned p2p_wait, p2p_signal;
  int dmma_stagger;  // dense_dmma: pairs 4..7 request their first tile only when pairs 0..3's rows have landed
  int64_t N;
  int D;
  int split;
  int a_start, a_count;  // active set = order[a_start .. a_start + a_count)
  int i_lo, i_hi;        // active ranks processed by this GPU (an upper bound for grid sizing when `range` is set)
  const int2* range;     // multi-GPU: device-resident [i_lo, i_hi) of this rank for this (step, split), or null
  // multi-GPU (P2P, dense_dmma): per (step, split) the owned active ranks with LOCAL partners first -- tile t
  // takes active ranks aperm[a_start + i_lo + 8 t ..]; null: natural order.  Same layout as `order`.
  const int32_t* aperm;
  int c_start[3], c_count[3];  // snooker: the three complement sets (ascending j != split)
  uint64_t seed, step;
  double p0, p1;  // stretch: a | de: g0, sigma | snooker: gammas
  ModelDev model;
  // optional taps (null unless debugging is enabled)
  int64_t* tap_partners;  // [3, N]
  double* tap_scalar;     // [N]
  double* tap_u;          // [N]
  int64_t* tap_active;    // [N]
  long long* timeline;    // dense_dmma instrumentation: [SM][consumer][tile<=TL_TILES][TL_EVENTS] cycles, or null
  const double* qbuf;     // MOVE_PRECOMPUTED: proposals [a_count, D] written by a proposal kernel (moves_extra.cu)
};

// internal move kind of half_step_generic_kernel: the proposal of active rank i is row i of HalfStepArgs::qbuf and
// the Hastings factor is 0 (WalkMove walk.py:37, GaussianMove gaussian.py:104); order == nullptr: walker id = i
constexpr int MOVE_PRECOMPUTED = 100;

struct Engine;  // defined in capi.cu

// launch shape of one fused half-step, as eb_debug_launch_config reports it (field order = the ABI's)
enum : int { SHAPE_NONE = 0, SHAPE_GENERIC = 1, SHAPE_TMA_ROWS = 2, SHAPE_DENSE_DMMA = 3 };
struct LaunchShape {
  int64_t kernel;   // SHAPE_*
  int64_t width;    // tma_rows / dense_dmma: walkers per tile; generic: lanes per walker
  int64_t epl;      // tma_rows: 8 on the register path, else 0
  int64_t own_reg;  // tma_rows: own row in registers
  int64_t warps;    // tma_rows: warps per CTA; dense_dmma: consumer warps per CTA; generic: threads / 32
  int64_t threads;  // threads per CTA
  int64_t grid;     // CTAs
  int64_t tiles;    // tiles of the half-step (generic: active walkers, one per lane group)
};

// ---- kernel launchers (implemented in the .cu files) ----------------------
// ranges (nullable): [nsteps_chunk, MAX_SPLITS] int2 = active ranks of each set owned by walkers [w_lo, w_hi)
cudaError_t launch_split_tables(int32_t* order, const StepInfo* info_dev, int nsteps_chunk, int64_t N,
                                uint64_t seed, uint64_t step0, int64_t w_lo, int64_t w_hi, int2* ranges,
                                cudaStream_t st);
// multi-GPU: for every (step, split) of the chunk, the active ranks [i_lo, i_hi) this rank owns with up to
// front_cap walkers whose stretch partner lives on this rank moved to the front (stable) -- tiles built from the
// front need no NVLink traffic and no peer barrier, so a half-step starts computing while the barrier and the
// first remote rows are still in flight
cudaError_t launch_locality_tables(const int32_t* order, const StepInfo* info_dev, const int2* ranges, int nsteps_chunk,
                                   int64_t N, uint64_t seed, uint64_t step0, int64_t rows_per_rank, int rank,
                                   int front_cap, int32_t* aperm, cudaStream_t st);
// shape (nullable): receives the launch shape
cudaError_t launch_half_step_generic(int move_kind, const HalfStepArgs& a, cudaStream_t st,
                                     LaunchShape* shape = nullptr);
// TMA row-gather variant for the HBM-bound models (tma_rows.cu); *used == false: not applicable, use the generic one
// (long_rows: also take rows so long that only one walker per tile fits; own_reg: stretch rows of <= 512 bytes keep
// the own row in registers -- plain loads / stores -- and stage only the partner rows).  max_grid: most CTAs of the
// grid-strided launch (the SM count, or less to give each warp more tiles).  *shape: the launch shape when used.
cudaError_t launch_half_step_tma(int move_kind, const HalfStepArgs& a, int max_grid, bool long_rows, bool own_reg,
                                 cudaStream_t st, bool* used, LaunchShape* shape);
cudaError_t launch_logprob_generic(const ModelDev& m, const double* x, int64_t rows, int D, double* out,
                                   int* status, cudaStream_t st);
// specialised: stretch + dense Gaussian on FP64 tensor cores (DMMA).  Returns
// cudaErrorNotSupported when the shape is outside its envelope.
bool dense_dmma_supported(int D);
size_t dense_dmma_factor_doubles(int D);
void dense_dmma_pack_factor(const double* L, int D, double* packed);  // host
// log-probability of dense-Gaussian rows on the tensor pipe (same arithmetic as the half-step kernel);
// max_grid: most CTAs of the grid-strided launch
cudaError_t launch_logprob_dense_dmma(const ModelDev& m, int D, const double* x, int64_t rows, double* out,
                                      int* status, int max_grid, cudaStream_t st);
// one half-step of a persistent dense_dmma launch
struct HalfDesc {
  uint64_t step;       // sampler step index (Philox counter)
  int32_t order_step;  // which split table of the chunk (also indexes `range`)
  int32_t split;
  int32_t a_start, a_count;
};
// runs `nhalf` consecutive half-steps in ONE cooperative launch (grid barrier between them);
// a.order / a.range point at the chunk's table bases; d0 == descs[0] travels by value.  max_count bounds the active ranks per
// half-step (grid sizing).  gbar is a monotonic global counter, gbar_base its value at launch.
// `pdl`: launch as a programmatic dependent of the previous kernel in the stream (nhalf == 1 only; the caller
// guarantees that kernel is a dense_dmma launch of the same run).  max_grid: most CTAs (at most the SM count:
// a cooperative launch needs every CTA resident).
cudaError_t launch_dense_dmma(const HalfStepArgs& a, const HalfDesc& d0, const HalfDesc* descs_dev, int nhalf,
                              int max_count,
                              unsigned long long* gbar, unsigned long long gbar_base, int max_grid, bool pdl,
                              LaunchShape* shape, cudaStream_t st);

// ---- proposal generators of WalkMove / GaussianMove (moves_extra.cu) ----------------------------
// acc = [S1 | S2] moment sums about a shift over n rows -> cov (np.cov) -> thresholded lower Cholesky factor L
cudaError_t launch_cov_chol(const double* acc, double n, int D, double* cov, double* L, cudaStream_t st);
cudaError_t launch_walk_shared_propose(const HalfStepArgs& a, const double* L, double* qbuf, cudaStream_t st);
bool walk_subset_supported(int D, int s0);
cudaError_t launch_walk_subset_propose(const HalfStepArgs& a, int s0, double* qbuf, cudaStream_t st);
cudaError_t launch_gaussian_shift(const double* L, int D, double f, uint64_t seed, uint64_t step, double* v,
                                  cudaStream_t st);
cudaError_t launch_gaussian_propose(const double* x0, int64_t row0, int64_t nrows, int D, int form, const double* scale,
                                    double f, int mode, int seq_dim, uint64_t seed, uint64_t step, double* qbuf,
                                    cudaStream_t st);

// ---- chain analysis (analysis.cu) ------------------------------------------------------------
// column means of X[nrows, D] (fixed summation order); status (nullable) gets the non-finite flags
cudaError_t launch_colmean(const double* X, int64_t nrows, int D, double* mean, int* status, cudaStream_t st);
// acc[D + D*D] += [sum(x - shift), (x - shift)^T (x - shift)] over the rows of X (DMMA; D <= 1024);
// partial: scratch of moments_partial_bytes(D, sm_count)
size_t moments_partial_bytes(int D, int sm_count);
// rowidx (nullable): row r of the set is walker rowidx[r < skip_start ? r : r + skip_count]
cudaError_t launch_moments(const double* X, int64_t nrows, int D, const double* shift, double* partial, double* acc,
                           int sm_count, cudaStream_t st, const int32_t* rowidx = nullptr, int skip_start = 0,
                           int skip_count = 0);

// walker-averaged normalised autocorrelation function (autocorr.py:21-46,101-107), slab by slab
int acf_fft_length(size_t n_t);
size_t acf_bytes_per_series(size_t n_t);
cudaError_t launch_acf_twiddles(double2* tw, int M, cudaStream_t st);
cudaError_t launch_acf_slab(const double* xin, int n_t, int wb, int nd, int M, const double2* tw, double2* z,
                            double* mean, double* f, cudaStream_t st);
cudaError_t launch_acf_scale(double* f, size_t n, double scale, cudaStream_t st);

inline int lanes_per_walker(int D) {
  int g = 4;
  while (g < 32 && g * 4 < D) g <<= 1;
  return g;
}

}  // namespace eb
