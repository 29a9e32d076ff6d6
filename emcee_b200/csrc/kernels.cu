// Split tables, the generic fused half-step kernel (any ndim / move / model) and
// the stand-alone log-probability kernel.
//
// Reference semantics implemented here (file:line relative to the reference):
//   split assignment + per-split gather order ... moves/red_blue.py:76-87
//   StretchMove.get_proposal ..................... moves/stretch.py:26-33
//   DEMove.get_proposal .......................... moves/de.py:40-64
//   DESnookerMove.get_proposal ................... moves/de_snooker.py:31-46
//   compute_log_prob guards ...................... ensemble.py:476-479,550-551
//   accept + update .............................. moves/red_blue.py:96-104, moves/move.py:29-34
#include <math.h>

#include "engine.cuh"
#include "rowops.cuh"

namespace eb {

// ===========================================================================
// split tables: order[] = walker ids grouped by set (ascending inside a set)
// ===========================================================================
// One block per step.  inds[w] = (randomize ? pi_step(w) : w) % P reproduces
// ``inds = arange(N) % P; shuffle(inds)`` (red_blue.py:77-80) with the keyed
// permutation of DESIGN.md; the stable partition of walkers by inds[] gives the
// ascending-walker order the boolean-mask gathers of red_blue.py:85 produce.
__global__ void __launch_bounds__(TABLE_THREADS) split_table_kernel(int32_t* __restrict__ order_base,
                                                                    const StepInfo* __restrict__ info,
                                                                    int64_t N, uint64_t seed,
                                                                    uint64_t step0, int64_t w_lo, int64_t w_hi,
                                                                    int2* __restrict__ ranges) {
  __shared__ int base[MAX_SPLITS];
  __shared__ int own_lo[MAX_SPLITS], own_hi[MAX_SPLITS];  // set members below w_lo / w_hi
  __shared__ int chunk_tot[MAX_SPLITS];
  __shared__ int warp_off[MAX_SPLITS][32];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint64_t step = step0 + blockIdx.x;
  const int P = info[blockIdx.x].nsplits;
  const bool randomize = info[blockIdx.x].randomize != 0;
  int32_t* order = order_base + (size_t)blockIdx.x * (size_t)N;

  if (tid < P) {
    // set j holds the walkers with inds == j: count_j = #{w < N : w % P == j}
    int64_t s = 0;
    for (int j = 0; j < tid; ++j) s += (N - j + P - 1) / P;
    base[tid] = (int)s;
    own_lo[tid] = 0;
    own_hi[tid] = 0;
  }
  const FeistelKeys fk = feistel_keys(seed, step);
  const int h = feistel_half_bits((uint64_t)N);
  __syncthreads();

  for (int64_t c0 = 0; c0 < N; c0 += TABLE_THREADS) {
    const int64_t w = c0 + tid;
    const bool valid = w < N;
    int sid = -1;
    if (valid) sid = (int)((randomize ? split_permute((uint64_t)w, (uint64_t)N, h, fk) : (uint64_t)w) % (uint64_t)P);
    int my_prefix = 0;
    for (int j = 0; j < P; ++j) {
      const unsigned b = __ballot_sync(0xffffffffu, sid == j);
      if (sid == j) my_prefix = __popc(b & ((1u << lane) - 1u));
      if (lane == 0) warp_off[j][warp] = __popc(b);
      if (ranges != nullptr) {  // multi-GPU: how many members of set j precede this rank's row block / its end
        const unsigned bl = __ballot_sync(0xffffffffu, sid == j && w < w_lo);
        const unsigned bh = __ballot_sync(0xffffffffu, sid == j && w < w_hi);
        if (lane == 0) {
          if (bl) atomicAdd(&own_lo[j], __popc(bl));
          if (bh) atomicAdd(&own_hi[j], __popc(bh));
        }
      }
    }
    __syncthreads();
    if (warp < P) {
      const int v = warp_off[warp][lane];
      int incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      warp_off[warp][lane] = incl - v;
      if (lane == 31) chunk_tot[warp] = incl;
    }
    __syncthreads();
    if (valid) order[base[sid] + warp_off[sid][warp] + my_prefix] = (int32_t)w;
    __syncthreads();
    if (tid < P) base[tid] += chunk_tot[tid];
    __syncthreads();
  }
  if (ranges != nullptr && tid < P) ranges[(size_t)blockIdx.x * MAX_SPLITS + tid] = make_int2(own_lo[tid], own_hi[tid]);
}

cudaError_t launch_split_tables(int32_t* order, const StepInfo* info_dev, int nsteps_chunk, int64_t N,
                                uint64_t seed, uint64_t step0, int64_t w_lo, int64_t w_hi, int2* ranges,
                                cudaStream_t st) {
  split_table_kernel<<<nsteps_chunk, TABLE_THREADS, 0, st>>>(order, info_dev, N, seed, step0, w_lo, w_hi, ranges);
  return cudaGetLastError();
}

// ===========================================================================
// locality tables (multi-GPU): owned active ranks, partner-local first
// ===========================================================================
// One block per (step of the chunk, split).  The stretch partner of active rank i is a pure function of
// (seed, step, split, i) and of the split table (stretch.py:32, DESIGN.md draw specification), so the order
// can be tabulated ahead for a whole chunk of steps like the split tables themselves.
__global__ void __launch_bounds__(TABLE_THREADS) locality_table_kernel(const int32_t* __restrict__ order_base,
                                                                       const StepInfo* __restrict__ info,
                                                                       const int2* __restrict__ ranges, int64_t N,
                                                                       uint64_t seed, uint64_t step0,
                                                                       int64_t rows_per_rank, int rank, int front_cap,
                                                                       int32_t* __restrict__ aperm_base) {
  __shared__ int warp_cnt[2][32], loc_cnt[32];
  __shared__ int base_sh[2], nfront_sh, seen_local_sh;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int P = info[blockIdx.x].nsplits, split = blockIdx.y;
  if (split >= P) return;
  const uint64_t step = step0 + blockIdx.x;
  const int32_t* order = order_base + (size_t)blockIdx.x * (size_t)N;
  int32_t* aperm = aperm_base + (size_t)blockIdx.x * (size_t)N;
  int a_start = 0;
  for (int j = 0; j < split; ++j) a_start += (int)((N - j + P - 1) / P);
  const int a_count = (int)((N - split + P - 1) / P);
  const int2 rg = ranges[(size_t)blockIdx.x * MAX_SPLITS + split];
  const int i_lo = rg.x, i_hi = rg.y;
  const int64_t Nc = N - a_count;
  auto is_local = [&](int i) -> bool {
    const u32x4 A = draw_words(seed, step, (uint32_t)split, TAG_PROP_A, (uint32_t)i);
    const int64_t r = (int64_t)bounded64(A.z, A.w, (uint64_t)Nc);  // stretch.py:32
    const int64_t wp = order[r < a_start ? r : r + a_count];
    return wp / rows_per_rank == rank;
  };
  // pass 1: how many owned active ranks have a local partner; at most `front_cap` of them (one tile per consumer
  // warp of the grid: the first round) move to the front, the rest of the list keeps its natural mix of local
  // and remote partners -- an all-remote tail would saturate the NVLink ports later instead
  int mine = 0;
  for (int i = i_lo + tid; i < i_hi; i += TABLE_THREADS) mine += is_local(i) ? 1 : 0;
  for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
  if (lane == 0) warp_cnt[0][warp] = mine;
  __syncthreads();
  if (tid == 0) {
    int tot = 0;
    for (int k = 0; k < TABLE_THREADS / 32; ++k) tot += warp_cnt[0][k];
    nfront_sh = tot < front_cap ? tot : front_cap;
    base_sh[0] = 0;          // next slot of the front group
    base_sh[1] = nfront_sh;  // next slot of the rest
    seen_local_sh = 0;       // local partners met so far (in natural order)
  }
  __syncthreads();
  // pass 2: stable two-way partition, chunk by chunk: front = the first nfront local-partner walkers
  for (int c0 = i_lo; c0 < i_hi; c0 += TABLE_THREADS) {
    const int i = c0 + tid;
    const bool valid = i < i_hi;
    const bool loc = valid && is_local(i);
    // rank of this walker among the local-partner ones
    const unsigned bloc = __ballot_sync(0xffffffffu, loc);
    if (lane == 0) warp_cnt[0][warp] = __popc(bloc);
    __syncthreads();
    int lrank = seen_local_sh + __popc(bloc & ((1u << lane) - 1u));
    for (int k = 0; k < warp; ++k) lrank += warp_cnt[0][k];
    const bool front = loc && lrank < nfront_sh;
    __syncthreads();
    const unsigned bf = __ballot_sync(0xffffffffu, front);
    const unsigned br = __ballot_sync(0xffffffffu, valid && !front);
    if (lane == 0) {
      warp_cnt[0][warp] = __popc(bf);
      warp_cnt[1][warp] = __popc(br);
      loc_cnt[warp] = __popc(bloc);
    }
    __syncthreads();
    int off = 0;
    const int grp = front ? 0 : 1;
    for (int k = 0; k < warp; ++k) off += warp_cnt[grp][k];
    const unsigned b = front ? bf : br;
    if (valid) aperm[a_start + i_lo + base_sh[grp] + off + __popc(b & ((1u << lane) - 1u))] = i;
    __syncthreads();
    if (tid < 2) {
      int tot = 0;
      for (int k = 0; k < TABLE_THREADS / 32; ++k) tot += warp_cnt[tid][k];
      base_sh[tid] += tot;
    } else if (tid == 2) {
      int tot = 0;
      for (int k = 0; k < TABLE_THREADS / 32; ++k) tot += loc_cnt[k];
      seen_local_sh += tot;
    }
    __syncthreads();
  }
}

cudaError_t launch_locality_tables(const int32_t* order, const StepInfo* info_dev, const int2* ranges, int nsteps_chunk,
                                   int64_t N, uint64_t seed, uint64_t step0, int64_t rows_per_rank, int rank,
                                   int front_cap, int32_t* aperm, cudaStream_t st) {
  locality_table_kernel<<<dim3(nsteps_chunk, MAX_SPLITS), TABLE_THREADS, 0, st>>>(order, info_dev, ranges, N, seed, step0,
                                                                                 rows_per_rank, rank, front_cap, aperm);
  return cudaGetLastError();
}

// ===========================================================================
// generic fused half-step: proposal + log-prob + accept + update
// ===========================================================================
// G lanes per active walker; the proposal row is staged in shared memory
// (rows_per_group rows of D doubles per group).
template <int MOVE, int MODEL>
__global__ void __launch_bounds__(256) half_step_generic_kernel(const HalfStepArgs a, const int G) {
  extern __shared__ double smem[];
  constexpr int NROWS = (MOVE == EB_MOVE_SNOOKER ? 4 : 1) + (MODEL == EB_MODEL_GAUSS_DENSE ? 1 : 0);
  const int D = a.D;
  const int groups = blockDim.x / G;
  const int gid = threadIdx.x / G, g = threadIdx.x % G;
  const int lane = threadIdx.x & 31;
  const unsigned mask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));
  const int i_lo = a.range ? a.range->x : a.i_lo;
  const int i_hi = a.range ? a.range->y : a.i_hi;
  const int64_t i = (int64_t)i_lo + (int64_t)blockIdx.x * groups + gid;
  if (i >= i_hi) return;  // whole groups leave together

  double* q = smem + (size_t)gid * NROWS * D;
  double* xc = q + (size_t)(NROWS - 1) * D;  // centred row (dense model only)
  const int64_t w = a.order ? (int64_t)a.order[a.a_start + i] : i;  // no table: the active set is every walker (MHMove)
  const double* s_row = a.coords + (size_t)w * D;  // the active walker is always local

  const u32x4 A = draw_words(a.seed, a.step, (uint32_t)a.split, TAG_PROP_A, (uint32_t)i);
  double factor = 0.0, tap_scalar = 0.0;
  int64_t pw[3] = {-1, -1, -1};

  if (MOVE == EB_MOVE_STRETCH) {
    const int64_t Nc = a.N - a.a_count;
    // stretch.py:30  zz = ((a - 1) * u + 1) ** 2 / a   (each op rounded once)
    const double t = __dadd_rn(__dmul_rn(__dsub_rn(a.p0, 1.0), u53(A.x, A.y)), 1.0);
    const double zz = __ddiv_rn(__dmul_rn(t, t), a.p0);
    // stretch.py:32  rint ; complement rank -> walker id
    const int64_t r = (int64_t)bounded64(A.z, A.w, (uint64_t)Nc);
    pw[0] = a.order[r < a.a_start ? r : r + a.a_count];
    const double* c_row = row_ptr(a, pw[0]);
    for (int e = g; e < D; e += G) {
      const double s = s_row[e], c = c_row[e];
      // stretch.py:33  q = c - (c - s) * zz   (no FMA contraction)
      const double v = __dsub_rn(c, __dmul_rn(__dsub_rn(c, s), zz));
      q[e] = v;
      if (!isfinite(v)) flag_nonfinite(v, a.status);
    }
    factor = __dmul_rn((double)D - 1.0, log(zz));  // stretch.py:31
    tap_scalar = zz;
  } else if (MOVE == EB_MOVE_DE) {
    const uint64_t Nc = (uint64_t)(a.N - a.a_count);
    const uint64_t m = bounded64(A.x, A.y, Nc * (Nc - 1));  // de.py:49
    uint64_t r0, r1;
    de_pair_decode(m, Nc, r0, r1);  // de.py:67-77
    pw[0] = a.order[(int64_t)r0 < a.a_start ? (int64_t)r0 : (int64_t)r0 + a.a_count];
    pw[1] = a.order[(int64_t)r1 < a.a_start ? (int64_t)r1 : (int64_t)r1 + a.a_count];
    const u32x4 B = draw_words(a.seed, a.step, (uint32_t)a.split, TAG_PROP_B, (uint32_t)i);
    const double n = sqrt(-2.0 * log(1.0 - u53(B.x, B.y))) * cos(6.283185307179586 * u53(B.z, B.w));
    const double gamma = __dmul_rn(a.p0, __dadd_rn(1.0, __dmul_rn(a.p1, n)));  // de.py:56
    const double* c0 = row_ptr(a, pw[0]);
    const double* c1 = row_ptr(a, pw[1]);
    for (int e = g; e < D; e += G) {
      // de.py:53,62  q = s + gamma * (c[p1] - c[p0])
      const double v = __dadd_rn(s_row[e], __dmul_rn(gamma, __dsub_rn(c1[e], c0[e])));
      q[e] = v;
      if (!isfinite(v)) flag_nonfinite(v, a.status);
    }
    tap_scalar = gamma;
  } else if (MOVE == MOVE_PRECOMPUTED) {
    // WalkMove / GaussianMove: the proposal was written by its own kernel (moves_extra.cu); factors = 0
    const double* qrow = a.qbuf + (size_t)(i - i_lo) * D;
    for (int e = g; e < D; e += G) {
      const double v = qrow[e];
      q[e] = v;
      if (!isfinite(v)) flag_nonfinite(v, a.status);
    }
  } else {  // EB_MOVE_SNOOKER
    const u32x4 B = draw_words(a.seed, a.step, (uint32_t)a.split, TAG_PROP_B, (uint32_t)i);
    int64_t cw[3];
    cw[0] = a.order[a.c_start[0] + (int64_t)bounded64(A.x, A.y, (uint64_t)a.c_count[0])];  // de_snooker.py:38
    cw[1] = a.order[a.c_start[1] + (int64_t)bounded64(A.z, A.w, (uint64_t)a.c_count[1])];
    cw[2] = a.order[a.c_start[2] + (int64_t)bounded64(B.x, B.y, (uint64_t)a.c_count[2])];
    // de_snooker.py:39  shuffle of the three rows -> one of 6 orders
    const int p = (int)bounded64(B.z, B.w, 6);
    const int i0 = p >> 1;                                 // 0,0,1,1,2,2
    const int rest0 = (i0 == 0) ? 1 : 0;                   // smaller of the remaining two
    const int rest1 = (i0 == 2) ? 1 : 2;                   // larger of the remaining two
    const int i1 = (p & 1) ? rest1 : rest0;
    const int i2 = (p & 1) ? rest0 : rest1;
    pw[0] = cw[i0];
    pw[1] = cw[i1];
    pw[2] = cw[i2];
    double* sS = q + (size_t)1 * D;  // rows: q | s | z | (z1 - z2 is streamed)
    double* sZ = q + (size_t)2 * D;
    double* sU = q + (size_t)3 * D;
    const double* z = row_ptr(a, pw[0]);
    const double* z1 = row_ptr(a, pw[1]);
    const double* z2 = row_ptr(a, pw[2]);
    double n2 = 0.0;
    for (int e = g; e < D; e += G) {
      const double s = s_row[e], zz_ = z[e];
      const double d = __dsub_rn(s, zz_);  // de_snooker.py:41 delta
      sS[e] = s;
      sZ[e] = zz_;
      sU[e] = d;
      n2 = fma(d, d, n2);
    }
    const double norm = sqrt(group_sum(n2, G, mask));  // de_snooker.py:42
    double d1 = 0.0, d2 = 0.0;
    for (int e = g; e < D; e += G) {
      const double u = __ddiv_rn(sU[e], norm);  // de_snooker.py:43
      sU[e] = u;
      d1 = fma(u, z1[e], d1);
      d2 = fma(u, z2[e], d2);
    }
    d1 = group_sum(d1, G, mask);
    d2 = group_sum(d2, G, mask);
    const double dd = __dsub_rn(d1, d2);
    double m2 = 0.0;
    for (int e = g; e < D; e += G) {
      // de_snooker.py:44  q = s + u * gammas * (u.z1 - u.z2)
      const double v = __dadd_rn(sS[e], __dmul_rn(__dmul_rn(sU[e], a.p0), dd));
      q[e] = v;
      if (!isfinite(v)) flag_nonfinite(v, a.status);
      const double dq = __dsub_rn(v, sZ[e]);
      m2 = fma(dq, dq, m2);
    }
    const double qn = sqrt(group_sum(m2, G, mask));
    factor = __dmul_rn((double)D - 1.0, __dsub_rn(log(qn), log(norm)));  // de_snooker.py:45-46
    tap_scalar = norm;
  }
  __syncwarp(mask);

  // red_blue.py:93 -> ensemble.py:458-553
  const double lp_new = model_logprob<MODEL>(q, xc, D, g, G, mask, a.model);
  if (isnan(lp_new) && g == 0) atomicOr(a.status, FLAG_NAN_LOGPROB);

  // red_blue.py:96-101
  const u32x4 U = draw_words(a.seed, a.step, (uint32_t)a.split, TAG_ACCEPT, (uint32_t)i);
  const double u_acc = u53(U.x, U.y);
  const double lnpdiff = __dsub_rn(__dadd_rn(factor, lp_new), a.logp[w]);
  const bool acc = lnpdiff > log(u_acc);

  // red_blue.py:103-104 -> move.py:29-34
  if (acc) {
    double* dst = a.coords + (size_t)w * D;
    for (int e = g; e < D; e += G) dst[e] = q[e];
  }
  if (g == 0) {
    if (acc) {
      a.logp[w] = lp_new;
      a.nacc[w] += 1ull;
    }
    a.accepted[w] = acc ? 1 : 0;
    if (a.tap_scalar != nullptr) {
      a.tap_partners[i] = pw[0];
      a.tap_partners[a.N + i] = pw[1];
      a.tap_partners[2 * a.N + i] = pw[2];
      a.tap_scalar[i] = tap_scalar;
      a.tap_u[i] = u_acc;
      a.tap_active[i] = w;
    }
  }
}

template <int MOVE, int MODEL>
static cudaError_t launch_generic_t(const HalfStepArgs& a, cudaStream_t st, LaunchShape* shape) {
  const int G = lanes_per_walker(a.D);
  constexpr int NROWS = (MOVE == EB_MOVE_SNOOKER ? 4 : 1) + (MODEL == EB_MODEL_GAUSS_DENSE ? 1 : 0);
  int threads = 256;
  size_t smem = (size_t)(threads / G) * NROWS * a.D * sizeof(double);
  while (smem > 200 * 1024 && threads > G) {
    threads >>= 1;
    smem = (size_t)(threads / G) * NROWS * a.D * sizeof(double);
  }
  if (smem > 200 * 1024) return cudaErrorInvalidConfiguration;
  const int groups = threads / G;
  const int64_t count = (int64_t)a.i_hi - a.i_lo;
  const unsigned grid = count > 0 ? (unsigned)((count + groups - 1) / groups) : 0u;
  if (shape) *shape = LaunchShape{SHAPE_GENERIC, G, 0, 0, threads / 32, threads, grid, count > 0 ? count : 0};
  if (count <= 0) return cudaSuccess;
  auto kern = half_step_generic_kernel<MOVE, MODEL>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  kern<<<grid, threads, smem, st>>>(a, G);
  return cudaGetLastError();
}

template <int MOVE>
static cudaError_t launch_generic_m(const HalfStepArgs& a, cudaStream_t st, LaunchShape* shape) {
  switch (a.model.kind) {
    case EB_MODEL_GAUSS_ISO:
      return launch_generic_t<MOVE, EB_MODEL_GAUSS_ISO>(a, st, shape);
    case EB_MODEL_GAUSS_DENSE:
      return launch_generic_t<MOVE, EB_MODEL_GAUSS_DENSE>(a, st, shape);
    case EB_MODEL_ROSENBROCK:
      return launch_generic_t<MOVE, EB_MODEL_ROSENBROCK>(a, st, shape);
    case EB_MODEL_RING:
      return launch_generic_t<MOVE, EB_MODEL_RING>(a, st, shape);
  }
  return cudaErrorInvalidValue;
}

cudaError_t launch_half_step_generic(int move_kind, const HalfStepArgs& a, cudaStream_t st, LaunchShape* shape) {
  switch (move_kind) {
    case EB_MOVE_STRETCH:
      return launch_generic_m<EB_MOVE_STRETCH>(a, st, shape);
    case EB_MOVE_DE:
      return launch_generic_m<EB_MOVE_DE>(a, st, shape);
    case EB_MOVE_SNOOKER:
      return launch_generic_m<EB_MOVE_SNOOKER>(a, st, shape);
    case MOVE_PRECOMPUTED:
      return launch_generic_m<MOVE_PRECOMPUTED>(a, st, shape);
  }
  return cudaErrorInvalidValue;
}

// ===========================================================================
// stand-alone log-probability (compute_log_prob, initial state)
// ===========================================================================
template <int MODEL>
__global__ void __launch_bounds__(256) logprob_generic_kernel(const ModelDev m, const double* __restrict__ x,
                                                              int64_t rows, int D, double* __restrict__ out,
                                                              int* status, const int G) {
  extern __shared__ double smem[];
  constexpr int NROWS = 1 + (MODEL == EB_MODEL_GAUSS_DENSE ? 1 : 0);
  const int groups = blockDim.x / G;
  const int gid = threadIdx.x / G, g = threadIdx.x % G;
  const int lane = threadIdx.x & 31;
  const unsigned mask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));
  const int64_t r = (int64_t)blockIdx.x * groups + gid;
  if (r >= rows) return;
  double* q = smem + (size_t)gid * NROWS * D;
  double* xc = q + (size_t)(NROWS - 1) * D;
  const double* src = x + (size_t)r * D;
  for (int e = g; e < D; e += G) {
    const double v = src[e];
    q[e] = v;
    if (!isfinite(v)) flag_nonfinite(v, status);  // ensemble.py:476-479
  }
  __syncwarp(mask);
  const double lp = model_logprob<MODEL>(q, xc, D, g, G, mask, m);
  if (g == 0) {
    out[r] = lp;
    if (isnan(lp)) atomicOr(status, FLAG_NAN_LOGPROB);  // ensemble.py:550-551
  }
}

template <int MODEL>
static cudaError_t launch_logprob_t(const ModelDev& m, const double* x, int64_t rows, int D, double* out,
                                    int* status, cudaStream_t st) {
  const int G = lanes_per_walker(D);
  constexpr int NROWS = 1 + (MODEL == EB_MODEL_GAUSS_DENSE ? 1 : 0);
  int threads = 256;
  size_t smem = (size_t)(threads / G) * NROWS * D * sizeof(double);
  while (smem > 200 * 1024 && threads > G) {
    threads >>= 1;
    smem = (size_t)(threads / G) * NROWS * D * sizeof(double);
  }
  if (smem > 200 * 1024) return cudaErrorInvalidConfiguration;
  if (rows <= 0) return cudaSuccess;
  const int groups = threads / G;
  auto kern = logprob_generic_kernel<MODEL>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  kern<<<(unsigned)((rows + groups - 1) / groups), threads, smem, st>>>(m, x, rows, D, out, status, G);
  return cudaGetLastError();
}

cudaError_t launch_logprob_generic(const ModelDev& m, const double* x, int64_t rows, int D, double* out,
                                   int* status, cudaStream_t st) {
  switch (m.kind) {
    case EB_MODEL_GAUSS_ISO:
      return launch_logprob_t<EB_MODEL_GAUSS_ISO>(m, x, rows, D, out, status, st);
    case EB_MODEL_GAUSS_DENSE:
      return launch_logprob_t<EB_MODEL_GAUSS_DENSE>(m, x, rows, D, out, status, st);
    case EB_MODEL_ROSENBROCK:
      return launch_logprob_t<EB_MODEL_ROSENBROCK>(m, x, rows, D, out, status, st);
    case EB_MODEL_RING:
      return launch_logprob_t<EB_MODEL_RING>(m, x, rows, D, out, status, st);
  }
  return cudaErrorInvalidValue;
}

}  // namespace eb
