// Fused half-step for the HBM-bound models (gauss_iso, ring, rosenbrock), any red-blue move,
// with the row gathers on the TMA engine.
//
// Reference semantics: identical to half_step_generic_kernel (kernels.cu): moves/red_blue.py:82-104,
// stretch.py:26-33, de.py:40-64, de_snooker.py:31-46, ensemble.py:476-479,550-551, move.py:29-34.
//
// Why a second kernel: these moves are pure row gathers -- a walker-step touches its own row
// and 1-3 random partner rows and does O(D) flops -- so the roof is HBM and what matters is how
// the rows travel.  Measured on this pool (eb_comm_probe, profiles/r01_nvlink_probe.txt): random
// 256-byte rows move at 1.3 TB/s with 16-byte loads and 4.3 TB/s as TMA bulk copies (0.28 vs
// 0.65 TB/s from a peer GPU).  So here every row is ONE cp.async.bulk into shared memory
// (completion on an mbarrier), accepted rows leave as ONE bulk store, and each warp runs a
// two-stage pipeline: the rows of tile k+1 are in flight while tile k is computed.
//
// Per-walker scalar work (two or three Philox blocks, the logs of the accept test, Box-Muller, the pair
// decode, the split-table lookups) is NOT done by the G lanes that share a walker's row: once per batch of
// G tiles (= 32 walkers) every lane does it for ONE walker, and the tile loop fetches what it needs with
// shuffles -- at 32-D that removes three quarters of the kernel's instructions (ncu: 964 -> ~500 per tile).
//
// Layout of a stage: [NR][R][D + pad] doubles -- NR rows per walker (own + partners), R walkers
// per tile, G = 32 / R lanes per walker; the pad (G doubles, 2 G on the register path) staggers consecutive
// walkers' rows across the banks so a warp-wide access costs the minimum number of wavefronts.
#include <math.h>

#include "engine.cuh"
#include "rowops.cuh"
#include "tma.cuh"

namespace eb {

namespace {

constexpr int TMA_MAX_THREADS = 512;  // 16 warps when the rows are short enough, else 8

template <int MOVE>
struct RowsPerWalker {
  static constexpr int value = MOVE == EB_MOVE_STRETCH ? 2 : (MOVE == EB_MOVE_DE ? 3 : 4);
};

// what one LANE keeps about one walker of the current batch of G tiles
struct WalkerMeta {
  int32_t w;       // active walker id, < 0 for the padding rows of a partial tile
  int32_t pw[3];   // partner walker ids (stretch: [0]; DE: p0, p1; snooker: z, z1, z2)
  double scalar;   // stretch: zz | DE: gamma
  double factor;   // stretch: (ndim - 1) log zz (stretch.py:31); else 0 (snooker's comes from the data)
  double log_u;    // log of the accept uniform (red_blue.py:100)
  double lp_old;   // current log-prob of the walker (red_blue.py:99); only this warp ever updates it
};

// EPL == 8: every lane owns 8 elements of its walker's row as four 16-byte chunks interleaved over the
// walker's lanes (chunk g + G k, k = 0..3: consecutive lanes read consecutive 16 bytes, no bank conflicts);
// needs ndim == 8 * lanes per walker, which covers 32-D at 8 walkers per tile, 128-D at 2, 256-D at 1.  Rows
// are read with 16-byte shared-memory loads into registers; the proposal, the log-probability and the snooker
// norms run on registers with fully unrolled loops.  EPL == 0: any even ndim, strided elements, run-time loops.
// OWN_REG (stretch, EPL == 8, rows of at most 512 bytes): the own row never touches shared memory -- it is read
// with four 16-byte global loads per lane one tile ahead, the proposal lives in registers and an accepted row is
// stored from them; only the partner rows travel by TMA.  For 256-byte rows the SM's TMA unit is the limiter
// (ncu: ~100 row copies/us against ~113 for a copy-only probe), and this takes two of the 2.3 row requests per
// walker-step off it.
template <int MOVE, int MODEL, int EPL, bool OWN_REG>
__global__ void __launch_bounds__(TMA_MAX_THREADS, 1) half_step_tma_kernel(const HalfStepArgs a, const int R) {
  static_assert(!OWN_REG || (MOVE == EB_MOVE_STRETCH && EPL == 8), "OWN_REG is the stretch register path");
  constexpr int NR = RowsPerWalker<MOVE>::value - (OWN_REG ? 1 : 0);  // rows per walker staged in shared memory
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int D = a.D;
  const int G = 32 / R;           // lanes per walker = tiles per batch
  // padded row stride (doubles): consecutive walkers' rows are staggered across the banks -- by G doubles for the
  // strided 8-byte accesses of the run-time path, by 2 G for the 16-byte chunks of the register path
  const int RS = D + (EPL == 8 ? 2 * G : G);
  const int stage_doubles = NR * R * RS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nwarps = blockDim.x >> 5;
  const int grp = lane / G, g = lane % G;
  const unsigned mask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));

  double* wbuf = reinterpret_cast<double*>(smem_raw) + (size_t)warp * 2 * stage_doubles;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)nwarps * 2 * stage_doubles * sizeof(double)) + 2 * warp;
  if (lane == 0) {
    mbar_init(bars + 0, 1);
    mbar_init(bars + 1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();

  const int i_lo = a.range ? a.range->x : a.i_lo;
  const int i_hi = a.range ? a.range->y : a.i_hi;
  const int64_t ntiles = ((int64_t)i_hi - i_lo + R - 1) / R;
  const int64_t tstride = (int64_t)gridDim.x * nwarps;
  const int64_t tile_first = (int64_t)blockIdx.x + (int64_t)gridDim.x * warp;  // SM-major deal, as dense_dmma
  const int64_t Nc = a.N - a.a_count;
  const unsigned row_bytes = (unsigned)(D * sizeof(double));

  // ---- draws and index lookups: lane l does walker (l % R) of tile (l / R) of batch kb -----------------
  auto prep_batch = [&](int64_t kb) -> WalkerMeta {
    WalkerMeta m;
    const int64_t tile = tile_first + (kb * G + lane / R) * tstride;
    int64_t i = (int64_t)i_lo + tile * R + (lane % R);
    const bool valid = tile < ntiles && i < i_hi;
    if (!valid) i = (int64_t)i_hi - 1;
    const u32x4 A = draw_words(a.seed, a.step, (uint32_t)a.split, TAG_PROP_A, (uint32_t)i);
    m.pw[0] = m.pw[1] = m.pw[2] = 0;
    m.scalar = 0.0;
    m.factor = 0.0;
    if (MOVE == EB_MOVE_STRETCH) {
      const double t = __dadd_rn(__dmul_rn(__dsub_rn(a.p0, 1.0), u53(A.x, A.y)), 1.0);  // stretch.py:30
      m.scalar = __ddiv_rn(__dmul_rn(t, t), a.p0);
      m.factor = __dmul_rn((double)D - 1.0, log(m.scalar));  // stretch.py:31
      const int64_t r = (int64_t)bounded64(A.z, A.w, (uint64_t)Nc);  // stretch.py:32
      m.pw[0] = __ldg(a.order + (r < a.a_start ? r : r + a.a_count));
    } else if (MOVE == EB_MOVE_DE) {
      const uint64_t mm = bounded64(A.x, A.y, (uint64_t)Nc * (uint64_t)(Nc - 1));  // de.py:49
      uint64_t r0, r1;
      de_pair_decode(mm, (uint64_t)Nc, r0, r1);  // de.py:67-77
      m.pw[0] = __ldg(a.order + ((int64_t)r0 < a.a_start ? (int64_t)r0 : (int64_t)r0 + a.a_count));
      m.pw[1] = __ldg(a.order + ((int64_t)r1 < a.a_start ? (int64_t)r1 : (int64_t)r1 + a.a_count));
      const u32x4 B = draw_words(a.seed, a.step, (uint32_t)a.split, TAG_PROP_B, (uint32_t)i);
      const double n = sqrt(-2.0 * log(1.0 - u53(B.x, B.y))) * cos(6.283185307179586 * u53(B.z, B.w));
      m.scalar = __dmul_rn(a.p0, __dadd_rn(1.0, __dmul_rn(a.p1, n)));  // de.py:56
    } else {
      const u32x4 B = draw_words(a.seed, a.step, (uint32_t)a.split, TAG_PROP_B, (uint32_t)i);
      int32_t cw[3];
      cw[0] = __ldg(a.order + a.c_start[0] + (int64_t)bounded64(A.x, A.y, (uint64_t)a.c_count[0]));  // de_snooker.py:38
      cw[1] = __ldg(a.order + a.c_start[1] + (int64_t)bounded64(A.z, A.w, (uint64_t)a.c_count[1]));
      cw[2] = __ldg(a.order + a.c_start[2] + (int64_t)bounded64(B.x, B.y, (uint64_t)a.c_count[2]));
      const int p = (int)bounded64(B.z, B.w, 6);  // de_snooker.py:39: one of the 6 row orders
      const int i0 = p >> 1;
      const int rest0 = (i0 == 0) ? 1 : 0, rest1 = (i0 == 2) ? 1 : 2;
      const int i1 = (p & 1) ? rest1 : rest0, i2 = (p & 1) ? rest0 : rest1;
      m.pw[0] = i0 == 0 ? cw[0] : (i0 == 1 ? cw[1] : cw[2]);
      m.pw[1] = i1 == 0 ? cw[0] : (i1 == 1 ? cw[1] : cw[2]);
      m.pw[2] = i2 == 0 ? cw[0] : (i2 == 1 ? cw[1] : cw[2]);
    }
    const int32_t w = __ldg(a.order + a.a_start + i);
    m.w = valid ? w : -(w + 1);  // keep the id (its rows are still fetched), flag it as padding
    const u32x4 U = draw_words(a.seed, a.step, (uint32_t)a.split, TAG_ACCEPT, (uint32_t)i);
    m.log_u = log(u53(U.x, U.y));
    m.lp_old = a.logp[w];
    return m;
  };
  // ---- launch the NR * R row copies of tile tb of a batch into a stage ---------------------------------
  auto issue = [&](const WalkerMeta& m, int tb, int stage) {
    double* buf = wbuf + (size_t)stage * stage_doubles;
    if (lane == 0) mbar_arrive_expect_tx(bars + stage, (unsigned)(NR * R) * row_bytes);
    __syncwarp();
    // copy c (< NR*R <= 32) is row j = c / R (+1 when the own row is not staged) of walker r = c % R; its ids
    // live in lane tb * R + r
    const int c = lane, j = c / R + (OWN_REG ? 1 : 0), r = c % R;
    const int src = (tb * R + r) & 31;
    const int wself = m.w >= 0 ? m.w : -(m.w + 1);
    const int src_self = __shfl_sync(0xffffffffu, wself, src);
    const int src_p0 = __shfl_sync(0xffffffffu, m.pw[0], src);
    const int src_p1 = __shfl_sync(0xffffffffu, m.pw[1], src);
    const int src_p2 = __shfl_sync(0xffffffffu, m.pw[2], src);
    if (c < NR * R) {
      const int64_t wr = j == 0 ? src_self : (j == 1 ? src_p0 : (j == 2 ? src_p1 : src_p2));
      const double* srcp = (j == 0) ? a.coords + (size_t)wr * D : row_ptr(a, wr);
      bulk_g2s(buf + ((size_t)(j - (OWN_REG ? 1 : 0)) * R + r) * RS, srcp, row_bytes, bars + stage);
    }
  };
  // OWN_REG: this lane's four 16-byte chunks of the own row of its group's walker in tile tb of a batch
  auto load_own = [&](const WalkerMeta& m, int tb, double (&v)[8]) {
    const int wsrc = __shfl_sync(0xffffffffu, m.w >= 0 ? m.w : -(m.w + 1), (tb * R + grp) & 31);
    const double* row = a.coords + (size_t)wsrc * D;
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const double2 t2 = __ldcg(reinterpret_cast<const double2*>(row + 2 * (g + G * kk)));
      v[2 * kk] = t2.x;
      v[2 * kk + 1] = t2.y;
    }
  };

  // this warp's k-th tile is tile_first + k * tstride; tiles come in batches of G (one walker per lane)
  WalkerMeta batch{}, batch_next{};
  double own_cur[8], own_next[8];  // OWN_REG: own rows of this tile / the next one
  if (tile_first < ntiles) {
    batch = prep_batch(0);
    issue(batch, 0, 0);
    if (OWN_REG) load_own(batch, 0, own_cur);
  }
  unsigned k = 0;
  for (int64_t tile = tile_first; tile < ntiles; tile += tstride, ++k) {
    const int stage = (int)(k & 1u);
    const int tb = (int)(k % (unsigned)G);
    double* buf = wbuf + (size_t)stage * stage_doubles;
    const bool has_next = tile + tstride < ntiles;
    if (has_next) {
      const bool crosses = tb + 1 == G;  // the next tile opens a new batch: tabulate it first
      if (crosses) batch_next = prep_batch((int64_t)(k + 1) / G);
      if (!OWN_REG) bulk_wait_read();  // the accepted rows of tile k-1 have left the other stage
      __syncwarp();
      if (crosses) {
        issue(batch_next, 0, stage ^ 1);
        if (OWN_REG) load_own(batch_next, 0, own_next);
      } else {
        issue(batch, tb + 1, stage ^ 1);
        if (OWN_REG) load_own(batch, tb + 1, own_next);
      }
    }
    // this group's walker: scalars from the lane that tabulated it
    const int me = (tb * R + grp) & 31;
    const int32_t cur_w = __shfl_sync(0xffffffffu, batch.w, me);
    const double cur_scalar = __shfl_sync(0xffffffffu, batch.scalar, me);
    const double cur_factor = __shfl_sync(0xffffffffu, batch.factor, me);
    const double cur_log_u = __shfl_sync(0xffffffffu, batch.log_u, me);
    const double cur_lp_old = __shfl_sync(0xffffffffu, batch.lp_old, me);
    mbar_wait(bars + stage, (k >> 1) & 1u);

    double* s = buf + ((size_t)0 * R + grp) * RS;  // own row, overwritten by the proposal (unused with OWN_REG)
    const bool valid = cur_w >= 0;
    const int64_t w = valid ? cur_w : -(cur_w + 1);
    double factor = cur_factor;

    double lp_new;
    double q_keep[8];  // OWN_REG: the proposal, kept for the store of an accepted row
    if constexpr (EPL == 8) {
      // ------- register path: this lane's elements are {2 (g + G k), 2 (g + G k) + 1}, k = 0..3 -------
      auto ld8 = [&](const double* row, double (&v)[8]) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const double2 t2 = *reinterpret_cast<const double2*>(row + 2 * (g + G * k));
          v[2 * k] = t2.x;
          v[2 * k + 1] = t2.y;
        }
      };
      double q[8];
      if (MOVE == EB_MOVE_STRETCH) {
        double sv[8], cv[8];
        if (OWN_REG) {
#pragma unroll
          for (int e = 0; e < 8; ++e) sv[e] = own_cur[e];
          ld8(buf + (size_t)grp * RS, cv);  // the only staged row of this walker
        } else {
          ld8(s, sv);
          ld8(buf + ((size_t)1 * R + grp) * RS, cv);
        }
        const double zz = cur_scalar;
#pragma unroll
        for (int e = 0; e < 8; ++e)  // stretch.py:33  q = c - (c - s) * zz   (each op rounded once)
          q[e] = __dsub_rn(cv[e], __dmul_rn(__dsub_rn(cv[e], sv[e]), zz));
      } else if (MOVE == EB_MOVE_DE) {
        double sv[8], c0[8], c1[8];
        ld8(s, sv);
        ld8(buf + ((size_t)1 * R + grp) * RS, c0);
        ld8(buf + ((size_t)2 * R + grp) * RS, c1);
        const double gamma = cur_scalar;
#pragma unroll
        for (int e = 0; e < 8; ++e)  // de.py:53,62  q = s + gamma * (c[p1] - c[p0])
          q[e] = __dadd_rn(sv[e], __dmul_rn(gamma, __dsub_rn(c1[e], c0[e])));
      } else {
        double sv[8], zv[8], u[8];
        ld8(s, sv);
        ld8(buf + ((size_t)1 * R + grp) * RS, zv);
        double n2 = 0.0;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          u[e] = __dsub_rn(sv[e], zv[e]);  // de_snooker.py:41
          n2 = fma(u[e], u[e], n2);
        }
        const double norm = sqrt(group_sum(n2, G, mask));  // de_snooker.py:42
        double d1 = 0.0, d2 = 0.0;
        {
          double z1[8], z2[8];
          ld8(buf + ((size_t)2 * R + grp) * RS, z1);
          ld8(buf + ((size_t)3 * R + grp) * RS, z2);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            u[e] = __ddiv_rn(u[e], norm);  // de_snooker.py:43
            d1 = fma(u[e], z1[e], d1);
            d2 = fma(u[e], z2[e], d2);
          }
        }
        d1 = group_sum(d1, G, mask);
        d2 = group_sum(d2, G, mask);
        const double dd = __dsub_rn(d1, d2);
        double m2 = 0.0;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          // de_snooker.py:44  q = s + u * gammas * (u.z1 - u.z2)
          q[e] = __dadd_rn(sv[e], __dmul_rn(__dmul_rn(u[e], a.p0), dd));
          const double dq = __dsub_rn(q[e], zv[e]);
          m2 = fma(dq, dq, m2);
        }
        const double qn = sqrt(group_sum(m2, G, mask));
        factor = __dmul_rn((double)D - 1.0, __dsub_rn(log(qn), log(norm)));  // de_snooker.py:45-46
      }
      if (OWN_REG) {
#pragma unroll
        for (int e = 0; e < 8; ++e) q_keep[e] = q[e];
      }
      bool bad = false;
#pragma unroll
      for (int e = 0; e < 8; ++e) bad |= !isfinite(q[e]);
      if (bad) {
#pragma unroll
        for (int e = 0; e < 8; ++e) flag_nonfinite(q[e], a.status);  // ensemble.py:476-479
      }
      if (!OWN_REG) {
#pragma unroll
        for (int k = 0; k < 4; ++k)  // the proposal replaces the own row: source of the bulk store
          *reinterpret_cast<double2*>(s + 2 * (g + G * k)) = make_double2(q[2 * k], q[2 * k + 1]);
      }
      // red_blue.py:93 -> ensemble.py:458-553: the registered models on registers (lane-sequential partial sums,
      // then the xor-shuffle reduction over the walker's lanes: the order depends only on ndim)
      double acc = 0.0;
      if (MODEL == EB_MODEL_GAUSS_ISO || MODEL == EB_MODEL_RING) {
#pragma unroll
        for (int e = 0; e < 8; ++e) acc = fma(q[e], q[e], acc);
        acc = group_sum(acc, G, mask);
        if (MODEL == EB_MODEL_GAUSS_ISO) {
          lp_new = -0.5 * acc;
        } else {
          const double d = sqrt(acc) - a.model.s0;
          lp_new = -(d * d) / (2.0 * a.model.s1 * a.model.s1);
        }
      } else {  // EB_MODEL_ROSENBROCK: x[e+1] of a chunk's second element is the next chunk's first element
        const int first = lane & ~(G - 1);  // first lane of this walker's group
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const double from_next_lane = __shfl_down_sync(mask, q[2 * k], 1);            // chunk g + 1 + G k
          const double from_first_lane = __shfl_sync(mask, q[k < 3 ? 2 * k + 2 : 0], first);  // chunk G (k + 1)
          const double x0 = q[2 * k], x1 = q[2 * k + 1];
          const double x2 = (g + 1 < G) ? from_next_lane : from_first_lane;
          {
            const double t1 = x1 - x0 * x0, u1 = a.model.s0 - x0;
            acc += a.model.s1 * (t1 * t1) + u1 * u1;
          }
          if (k < 3 || g + 1 < G) {  // (element ndim - 1 has no successor)
            const double t1 = x2 - x1 * x1, u1 = a.model.s0 - x1;
            acc += a.model.s1 * (t1 * t1) + u1 * u1;
          }
        }
        lp_new = -group_sum(acc, G, mask);
      }
    } else {
      if (MOVE == EB_MOVE_STRETCH) {
        const double* c = buf + ((size_t)1 * R + grp) * RS;
        const double zz = cur_scalar;
        for (int e = g; e < D; e += G) {
          const double sv = s[e], cv = c[e];
          // stretch.py:33  q = c - (c - s) * zz   (each op rounded once, no FMA contraction)
          const double v = __dsub_rn(cv, __dmul_rn(__dsub_rn(cv, sv), zz));
          s[e] = v;
          if (!isfinite(v)) flag_nonfinite(v, a.status);
        }
      } else if (MOVE == EB_MOVE_DE) {
        const double* c0 = buf + ((size_t)1 * R + grp) * RS;
        const double* c1 = buf + ((size_t)2 * R + grp) * RS;
        const double gamma = cur_scalar;
        for (int e = g; e < D; e += G) {
          // de.py:53,62  q = s + gamma * (c[p1] - c[p0])
          const double v = __dadd_rn(s[e], __dmul_rn(gamma, __dsub_rn(c1[e], c0[e])));
          s[e] = v;
          if (!isfinite(v)) flag_nonfinite(v, a.status);
        }
      } else {
        const double* z = buf + ((size_t)1 * R + grp) * RS;
        double* z1 = buf + ((size_t)2 * R + grp) * RS;  // becomes u
        const double* z2 = buf + ((size_t)3 * R + grp) * RS;
        double n2 = 0.0;
        for (int e = g; e < D; e += G) {
          const double d = __dsub_rn(s[e], z[e]);  // de_snooker.py:41
          n2 = fma(d, d, n2);
        }
        const double norm = sqrt(group_sum(n2, G, mask));  // de_snooker.py:42
        double d1 = 0.0, d2 = 0.0;
        for (int e = g; e < D; e += G) {
          const double u = __ddiv_rn(__dsub_rn(s[e], z[e]), norm);  // de_snooker.py:43
          d1 = fma(u, z1[e], d1);
          d2 = fma(u, z2[e], d2);
          z1[e] = u;
        }
        d1 = group_sum(d1, G, mask);
        d2 = group_sum(d2, G, mask);
        const double dd = __dsub_rn(d1, d2);
        double m2 = 0.0;
        for (int e = g; e < D; e += G) {
          // de_snooker.py:44  q = s + u * gammas * (u.z1 - u.z2)
          const double v = __dadd_rn(s[e], __dmul_rn(__dmul_rn(z1[e], a.p0), dd));
          s[e] = v;
          if (!isfinite(v)) flag_nonfinite(v, a.status);
          const double dq = __dsub_rn(v, z[e]);
          m2 = fma(dq, dq, m2);
        }
        const double qn = sqrt(group_sum(m2, G, mask));
        factor = __dmul_rn((double)D - 1.0, __dsub_rn(log(qn), log(norm)));  // de_snooker.py:45-46
      }
      __syncwarp(mask);

      // red_blue.py:93 -> ensemble.py:458-553
      lp_new = model_logprob<MODEL>(s, nullptr, D, g, G, mask, a.model);
    }
    if (isnan(lp_new) && g == 0) atomicOr(a.status, FLAG_NAN_LOGPROB);
    // red_blue.py:96-101
    const double lnpdiff = __dsub_rn(__dadd_rn(factor, lp_new), cur_lp_old);
    const bool acc = valid && (lnpdiff > cur_log_u);
    if constexpr (OWN_REG) {
      // red_blue.py:103-104 -> move.py:29-34: an accepted row is stored from the registers that hold the proposal
      if (acc) {
        double* dst = a.coords + (size_t)w * D;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          *reinterpret_cast<double2*>(dst + 2 * (g + G * kk)) = make_double2(q_keep[2 * kk], q_keep[2 * kk + 1]);
      }
      if (g == 0) {
        if (acc) {
          a.logp[w] = lp_new;
          atomicAdd(a.nacc + w, 1ull);
        }
        if (valid) a.accepted[w] = acc ? 1 : 0;
      }
      __syncwarp();  // every lane is done reading this stage before the next iteration refills it
#pragma unroll
      for (int e = 0; e < 8; ++e) own_cur[e] = own_next[e];
    } else {
      // red_blue.py:103-104 -> move.py:29-34: one bulk store per accepted row
      fence_async_smem();
      __syncwarp();
      if (g == 0) {
        if (acc) {
          bulk_s2g(a.coords + (size_t)w * D, s, row_bytes);
          a.logp[w] = lp_new;
          atomicAdd(a.nacc + w, 1ull);
        }
        if (valid) a.accepted[w] = acc ? 1 : 0;
      }
      bulk_commit();
    }
    if (tb + 1 == G) batch = batch_next;
  }
  // every accepted row has left shared memory AND reached global memory before the warp retires
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

template <int MOVE, int MODEL>
cudaError_t launch_tma_t(const HalfStepArgs& a, int max_grid, bool long_rows, bool own_rows_in_registers, cudaStream_t st,
                         bool* used, LaunchShape* shape) {
  constexpr int NR = RowsPerWalker<MOVE>::value;
  *used = false;
  const int D = a.D;
  if (D % 2 != 0) return cudaSuccess;  // rows must be multiples of 16 bytes for bulk copies
  // Latency is hidden by warps: 16 per SM when each one's two stages fit a 12 KB share of shared memory;
  // walkers per tile R = the largest power of two with NR*R <= 32 copies per stage that fits.  Rows so long
  // that only one walker per tile fits (e.g. 256-D DE / snooker) run with R = 1 and as many warps (>= 8) as
  // 200 KB hold -- `long_rows`; measured against the generic kernel in profiles/r02_hbm_kernels.md.
  auto warp_bytes = [&](int r) {
    const int pad = (D == 8 * (32 / r)) ? 2 * (32 / r) : 32 / r;  // the kernel's row stride (register path: 2 G)
    return (size_t)2 * NR * r * (D + pad) * sizeof(double);
  };
  int nwarps = 16;
  const size_t budget = (size_t)192 * 1024 / nwarps;
  int R = 0;
  for (int r = 16; r >= 2; r >>= 1)
    if (NR * r <= 32 && warp_bytes(r) <= budget) {
      R = r;
      break;
    }
  if (R == 0 && long_rows) {
    const size_t fit = ((size_t)200 * 1024) / warp_bytes(1);
    if (fit >= 8) {
      R = 1;
      nwarps = (int)(fit < 16 ? fit : 16);
    }
  }
  if (R == 0) return cudaSuccess;  // generic kernel
  const bool epl8 = D == 8 * (32 / R);  // 8 elements per lane: the register path
  // short rows (<= 512 B) of the stretch move: own rows by plain loads, only the partner rows on the TMA unit
  const bool own_reg = MOVE == EB_MOVE_STRETCH && epl8 && D <= 64 && own_rows_in_registers;
  const int nr_smem = NR - (own_reg ? 1 : 0);
  const size_t smem = (size_t)nwarps * warp_bytes(R) / NR * nr_smem + (size_t)nwarps * 2 * sizeof(uint64_t);
  const int64_t count = (int64_t)a.i_hi - a.i_lo;
  const int64_t ntiles = count > 0 ? (count + R - 1) / R : 0;
  const int64_t want = (ntiles + nwarps - 1) / nwarps;
  const int grid = (int)(want < max_grid ? want : max_grid);
  *shape = LaunchShape{SHAPE_TMA_ROWS, R, epl8 ? 8 : 0, own_reg ? 1 : 0, nwarps, 32 * nwarps, grid, ntiles};
  if (count <= 0) {
    *used = true;
    return cudaSuccess;
  }
  void (*kern)(const HalfStepArgs, const int) =
      epl8 ? half_step_tma_kernel<MOVE, MODEL, 8, false> : half_step_tma_kernel<MOVE, MODEL, 0, false>;
  if constexpr (MOVE == EB_MOVE_STRETCH) {
    if (own_reg) kern = half_step_tma_kernel<MOVE, MODEL, 8, true>;
  }
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kern<<<grid, 32 * nwarps, smem, st>>>(a, R);
  *used = true;
  return cudaGetLastError();
}

template <int MOVE>
cudaError_t launch_tma_m(const HalfStepArgs& a, int max_grid, bool long_rows, bool own_reg, cudaStream_t st, bool* used,
                         LaunchShape* shape) {
  switch (a.model.kind) {
    case EB_MODEL_GAUSS_ISO:
      return launch_tma_t<MOVE, EB_MODEL_GAUSS_ISO>(a, max_grid, long_rows, own_reg, st, used, shape);
    case EB_MODEL_ROSENBROCK:
      return launch_tma_t<MOVE, EB_MODEL_ROSENBROCK>(a, max_grid, long_rows, own_reg, st, used, shape);
    case EB_MODEL_RING:
      return launch_tma_t<MOVE, EB_MODEL_RING>(a, max_grid, long_rows, own_reg, st, used, shape);
  }
  *used = false;  // dense Gaussian outside the DMMA envelope: CUDA-core generic kernel
  return cudaSuccess;
}

}  // namespace

// Tries the TMA row-gather kernel; *used tells whether it took the half-step (otherwise the
// caller falls back to half_step_generic_kernel).
cudaError_t launch_half_step_tma(int move_kind, const HalfStepArgs& a, int max_grid, bool long_rows, bool own_reg,
                                 cudaStream_t st, bool* used, LaunchShape* shape) {
  switch (move_kind) {
    case EB_MOVE_STRETCH:
      return launch_tma_m<EB_MOVE_STRETCH>(a, max_grid, long_rows, own_reg, st, used, shape);
    case EB_MOVE_DE:
      return launch_tma_m<EB_MOVE_DE>(a, max_grid, long_rows, own_reg, st, used, shape);
    case EB_MOVE_SNOOKER:
      return launch_tma_m<EB_MOVE_SNOOKER>(a, max_grid, long_rows, own_reg, st, used, shape);
  }
  *used = false;
  return cudaErrorInvalidValue;
}

}  // namespace eb
