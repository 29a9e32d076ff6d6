// Fused half-step for StretchMove + dense Gaussian on the FP64 tensor pipe.
//
// Reference semantics: moves/red_blue.py:82-104 with moves/stretch.py:26-33 as the
// proposal and log_prob(x) = -0.5 (x-mu)^T A (x-mu) (document/plots/oned.py:17-18).
//
// Design (DESIGN.md "dense_dmma"):
//   * A = L L^T is factored once on the host; lp = -0.5 |L^T (q - mu)|^2, i.e. a
//     [walkers x D] x [D x D lower-triangular] product: only the blocks on or
//     below the diagonal are multiplied (D(D+1) instead of 2 D^2 flops).
//   * persistent CTAs, one per SM, warp specialised: 8 CONSUMER warps (two per SM
//     sub-partition -- what the FP64 tensor pipe needs to stay saturated when its B
//     operand streams from shared memory) and 8 PRODUCER warps, paired 1:1.
//   * producer p: Philox draws, order[] lookups, old log-prob, the two logs of the
//     accept test -> a small meta record in shared memory; 16 TMA bulk copies
//     (cp.async.bulk, one whole 8*D-byte row each: the active walker's row and its
//     partner's, possibly from a peer GPU over NVLink) into the pair's landing
//     slot, completion counted on an mbarrier; then the proposal
//     q = c - (c - s) z (bit-exact sub/mul/sub) written over the partner rows.
//   * consumer c: loads q into REGISTERS (lane (g,t) holds row g, columns
//     {8j+2t, 8j+2t+1}: the DMMA A fragments under a permutation of the contraction
//     index that is folded into the packing of L, so rows move as 16-byte vectors),
//     releases the slot (the producer refills it while the tile is on the tensor
//     pipe), runs mma.sync.m8n8k4.f64 against the packed factor in shared memory,
//     reduces |y|^2 over the 4 lanes of a row, applies the Metropolis test and
//     writes accepted rows straight from those registers.  A consumer does almost
//     nothing but DMMAs.
//   * tiles (8 walkers) are dealt SM-major, so every sub-partition gets the same count.
//   * one cooperative launch runs MANY half-steps (all splits of all steps up to the
//     next host-visible event): between half-steps the CTAs meet at a grid barrier on
//     a global counter instead of paying a kernel boundary (launch gap, re-staging of
//     the 70 KB factor, pipeline refill from cold).
#include <math.h>

#include "engine.cuh"
#include "tma.cuh"

namespace eb {

namespace {

constexpr int DMMA_CONSUMERS = 8;
constexpr int DMMA_THREADS = 64 * DMMA_CONSUMERS;  // consumers are warps 0..7, producers 8..15
constexpr int NI = 2;  // column tiles in flight per consumer (2*NI independent accumulator chains)

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__host__ __device__ constexpr int packed_blocks(int KB) { return KB * (KB + 1); }  // 2 * KB(KB+1)/2
// landing slot of one pair: [s|c][8 rows][D + 8] doubles; the +8 (64 B) row skew
// makes the 16-byte fragment accesses of 8 consecutive lanes hit 32 distinct banks
__host__ __device__ constexpr int row_stride(int KB) { return 8 * KB + 8; }

// what the producer hands to the consumer besides q (one record per tile, two in flight)
struct TileMeta {
  double factor[8];  // (ndim - 1) log zz                              (stretch.py:31)
  double log_u[8];   // log of the accept uniform                      (red_blue.py:100)
  double lp_old[8];  // current log-prob of the active walker          (red_blue.py:99)
  int32_t w[8];      // active walker id; < 0: padding row of a partial tile
};

template <int KB>
struct SmemLayout {
  static constexpr size_t L_doubles = (size_t)packed_blocks(KB) * 32;
  static constexpr size_t mu_doubles = 8 * KB;
  static constexpr size_t slot_doubles = 2 * 8 * row_stride(KB);
  static constexpr size_t off_mu = L_doubles;
  static constexpr size_t off_slots = off_mu + mu_doubles;
  static constexpr size_t off_meta = off_slots + DMMA_CONSUMERS * slot_doubles;  // in doubles
  static constexpr size_t meta_bytes = sizeof(TileMeta) * 2 * DMMA_CONSUMERS;
  static constexpr size_t off_bars_bytes = off_meta * sizeof(double) + meta_bytes;
  static constexpr int nbars = 1 + 3 * DMMA_CONSUMERS;
  static constexpr size_t off_abort_bytes = off_bars_bytes + nbars * sizeof(uint64_t);
  static constexpr size_t total_bytes = off_abort_bytes + 16;
};

// The tensor-pipe block of the stand-alone log-prob kernel: the same statements, in the same order, as
// the block inlined in the half-step kernel's consumer (kept inline there: its register allocation is
// tuned to the last register), so both produce bit-identical values for the same row: this lane's partial sum over its two columns of
// |L^T (q - mu)|^2 for the 8 rows of the warp's tile; q holds the lane's A fragments.
template <int KB, bool HAS_MEAN>
__device__ __forceinline__ double tile_sumsq(const double (&q)[2 * KB], const double* sL, const double* sMu, int lane,
                                             int t) {
  double rs = 0.0;
  const double* bptr = sL + 2 * lane;  // one 16-byte load feeds the two k-halves of a block pair
#pragma unroll
  for (int nb0 = 0; nb0 < KB; nb0 += NI) {
    double c[NI][2][2];
#pragma unroll
    for (int n = 0; n < NI; ++n) c[n][0][0] = c[n][0][1] = c[n][1][0] = c[n][1][1] = 0.0;
#pragma unroll
    for (int j = nb0; j < KB; ++j) {
      double x0 = q[2 * j + 0], x1 = q[2 * j + 1];
      if (HAS_MEAN) {
        const double2 m2 = *reinterpret_cast<const double2*>(sMu + 8 * j + 2 * t);
        x0 -= m2.x;
        x1 -= m2.y;
      }
#pragma unroll
      for (int n = 0; n < NI; ++n) {
        if (nb0 + n < KB && j >= nb0 + n) {
          const double2 b2 = *reinterpret_cast<const double2*>(bptr);
          dmma884(c[n][0][0], c[n][0][1], x0, b2.x);
          dmma884(c[n][1][0], c[n][1][1], x1, b2.y);
          bptr += 64;
        }
      }
    }
#pragma unroll
    for (int n = 0; n < NI; ++n) {
      const double y0 = c[n][0][0] + c[n][1][0], y1 = c[n][0][1] + c[n][1][1];
      rs = fma(y0, y0, rs);
      rs = fma(y1, y1, rs);
    }
  }
  return rs;
}

// grid-wide barrier between consecutive half-steps of one persistent launch: the
// consumers of every CTA publish "my writes of half-step h are out" on a global
// counter; producers wait for all CTAs before they read state for half-step h+1.
__device__ __forceinline__ bool grid_wait(const unsigned long long* counter, unsigned long long target, int* status) {
  const long long t0 = clock64();
  while (*reinterpret_cast<const volatile unsigned long long*>(counter) < target) {
    __nanosleep(32);
    if (clock64() - t0 > 60000000000ll) {  // ~30 s: never hang the GPU on a lost CTA
      atomicOr(status, FLAG_COMM_TIMEOUT);
      return false;
    }
  }
  __threadfence();
  return true;
}

// multi-GPU: lanes 0..nranks-1 of a warp wait until every peer has published `target` (or later) into
// this rank's flag array; false on timeout (a peer died).
__device__ __forceinline__ bool peer_wait(const unsigned* my_flags, int rank, int nranks, unsigned target, int lane,
                                          int* status) {
  bool ok = true;
  if (lane < nranks && lane != rank) {
    const volatile unsigned* f = my_flags + lane;
    const long long t0 = clock64();
    while ((int)(*f - target) < 0) {
      __nanosleep(64);
      if (clock64() - t0 > 60000000000ll) {  // ~30 s
        atomicOr(status, FLAG_COMM_TIMEOUT);
        ok = false;
        break;
      }
    }
  }
  __threadfence_system();
  return __all_sync(0xffffffffu, ok);
}

template <int KB, bool HAS_MEAN>
__global__ void __launch_bounds__(DMMA_THREADS, 1)
    half_step_dense_dmma_kernel(const HalfStepArgs a, const HalfDesc d0, const HalfDesc* __restrict__ descs,
                                const int nhalf, unsigned long long* gbar, const unsigned long long gbar_base) {
  constexpr int D = 8 * KB;
  constexpr int RS = row_stride(KB);
  using SL = SmemLayout<KB>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sL = reinterpret_cast<double*>(smem_raw);
  double* sMu = sL + SL::off_mu;
  double* sSlots = sL + SL::off_slots;
  TileMeta* sMeta = reinterpret_cast<TileMeta*>(sL + SL::off_meta);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + SL::off_bars_bytes);
  // CTA-wide abort flag: a producer that gives up on a lost peer / CTA sets it, every wait polls it, so all
  // warps leave and the host reports FLAG_COMM_TIMEOUT instead of the kernel spinning into a trap
  volatile int* sAbort = reinterpret_cast<volatile int*>(smem_raw + SL::off_abort_bytes);
  // multi-GPU: number of half-steps of this launch whose peer barrier this CTA has passed (written by the
  // producer of pair 0).  Tiles whose partners are all local start before it; remote fetches and every
  // store of an accepted row wait for it.
  volatile int* sPeers = sAbort + 1;
  uint64_t* barL = bars;                                  // packed factor landed
  uint64_t* barFull = bars + 1;                           // [pair] TMA: rows of a tile landed
  uint64_t* barReady = bars + 1 + DMMA_CONSUMERS;         // [pair] producer: proposal written
  uint64_t* barFree = bars + 1 + 2 * DMMA_CONSUMERS;      // [pair] consumer: slot may be refilled

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool is_producer = warp >= DMMA_CONSUMERS;
  const int pair = is_producer ? warp - DMMA_CONSUMERS : warp;
  const int g = lane >> 2, t = lane & 3;

  if (tid == 0) {
    *sAbort = 0;
    *sPeers = 0;
    mbar_init(barL, 1);
    for (int c = 0; c < DMMA_CONSUMERS; ++c) {
      mbar_init(barFull + c, 1);
      mbar_init(barReady + c, 1);
      mbar_init(barFree + c, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (HAS_MEAN)
    for (int k = tid; k < D; k += DMMA_THREADS) sMu[k] = a.model.params[k];
  __syncthreads();
  if (tid == 0) {  // one bulk copy brings the whole packed factor, once per launch
    constexpr unsigned bytes = (unsigned)(SL::L_doubles * sizeof(double));
    mbar_arrive_expect_tx(barL, bytes);
    bulk_g2s(sL, a.model.chol, bytes, barL);
  }

  const int64_t tstride = (int64_t)gridDim.x * DMMA_CONSUMERS;
  const int64_t tile0 = (int64_t)blockIdx.x + (int64_t)gridDim.x * pair;  // SM-major deal
  double* slot = sSlots + (size_t)pair * SL::slot_doubles;
  double* myS = slot + (size_t)g * RS + 2 * t;  // this lane's 16-byte chunks of row g
  double* myC = myS + 8 * RS;                   // partner row, later the proposal
  TileMeta* meta = sMeta + 2 * pair;
  const bool multi = a.p2p_peer_flags != nullptr;
  unsigned k = 0;  // tiles this pair has handled so far in the launch (mbarrier phase counter)

  if (is_producer) {
    // ================= producer: draws, lookups, TMA row gather, proposal =================
    // optional stamps of the LAST half-step, events 6..8 of the tile's record (cycles since this warp entered
    // the kernel): 6 rows requested, 7 rows landed, 8 proposal published
    const long long t_entry_p = clock64();
    long long* tlp = (a.timeline && lane == 0)
                         ? a.timeline + ((size_t)blockIdx.x * DMMA_CONSUMERS + pair) * TL_TILES * TL_EVENTS : nullptr;
    const double dm1 = (double)a.D - 1.0;
    const int row = lane & 7;
    // per-row quantities of one tile (every lane mirrors row lane & 7)
    struct Prep {
      int32_t w, wp;
      double zz, factor, log_u, lp_old;
      bool valid, remote;
    };
    for (int h = 0; h < nhalf; ++h) {
      const HalfDesc d = (h == 0) ? d0 : descs[h];  // the first one travels in the launch parameters
      const int32_t* order = a.order + (size_t)d.order_step * a.N;
      const int2 rg = a.range ? a.range[(size_t)d.order_step * MAX_SPLITS + d.split] : make_int2(0, d.a_count);
      const int i_lo = rg.x, i_hi = rg.y;
      const int64_t ntiles = ((int64_t)i_hi - i_lo + 7) >> 3;
      const int64_t Nc = a.N - d.a_count;
      // draws + index lookups: independent of the walker state, so they run ahead of the grid barrier
      const int32_t* aperm = a.aperm ? a.aperm + (size_t)d.order_step * a.N + d.a_start : nullptr;
      auto prep = [&](int64_t tile, bool with_lp) -> Prep {
        Prep p;
        int64_t i = (int64_t)i_lo + tile * 8 + row;
        p.valid = i < i_hi;
        if (!p.valid) i = (int64_t)i_hi - 1;
        if (aperm) i = __ldg(aperm + i);  // sharded: tiles are built partner-local first (locality_table_kernel)
        const u32x4 A = draw_words(a.seed, d.step, (uint32_t)d.split, TAG_PROP_A, (uint32_t)i);
        const double tt = __dadd_rn(__dmul_rn(__dsub_rn(a.p0, 1.0), u53(A.x, A.y)), 1.0);  // stretch.py:30
        p.zz = __ddiv_rn(__dmul_rn(tt, tt), a.p0);
        const int64_t r = (int64_t)bounded64(A.z, A.w, (uint64_t)Nc);  // stretch.py:32
        p.w = __ldg(order + d.a_start + i);
        p.wp = __ldg(order + (r < d.a_start ? r : r + d.a_count));
        const u32x4 U = draw_words(a.seed, d.step, (uint32_t)d.split, TAG_ACCEPT, (uint32_t)i);
        p.log_u = log(u53(U.x, U.y));
        p.factor = __dmul_rn(dm1, log(p.zz));  // stretch.py:31
        p.lp_old = with_lp ? a.logp[p.w] : 0.0;
        p.remote = multi && (p.wp / a.rows_per_rank != a.p2p_rank);
        return p;
      };
      // multi-GPU: the peer barrier of this half-step (every rank has finished the previous one).  Pair 0's
      // producer waits on the peer flags and publishes the result to the CTA; the others wait for that.
      auto peers_ready = [&]() -> bool {
        if (!multi || *sPeers > h) return true;
        if (pair == 0) {
          if (!peer_wait(a.p2p_my_flags, a.p2p_rank, a.p2p_nranks, a.p2p_wait + (unsigned)h, lane, a.status)) {
            *sAbort = 1;
            return false;
          }
          __syncwarp();
          if (lane == 0) *sPeers = h + 1;
        } else {
          while (*sPeers <= h) {
            if (*sAbort) return false;
            __nanosleep(64);
          }
        }
        asm volatile("fence.proxy.async;" ::: "memory");  // peers' generic-proxy writes -> our TMA reads
        return true;
      };
      // publish the meta record and launch the 16 row copies of one tile into the landing slot
      auto issue = [&](Prep& p, int par, bool load_lp) -> bool {
        if (__any_sync(0xffffffffu, p.remote) && !peers_ready()) return false;
        if (lane == 0) mbar_arrive_expect_tx(barFull + pair, 16u * D * (unsigned)sizeof(double));
        __syncwarp();
        if (lane < 16) {
          const bool partner = lane >= 8;
          const int64_t wr = partner ? (int64_t)p.wp : (int64_t)p.w;
          const double* base =
              (partner && a.peer_coords != nullptr) ? a.peer_coords[wr / a.rows_per_rank] : a.coords;
          bulk_g2s(slot + (size_t)(partner ? 8 : 0) * RS + (size_t)row * RS, base + (size_t)wr * D,
                   (unsigned)(D * sizeof(double)), barFull + pair);
        }
        if (load_lp) p.lp_old = a.logp[p.w];  // behind the row copies: off the post-barrier critical path
        TileMeta* m = meta + par;
        if (lane < 8) {
          m->factor[row] = p.factor;
          m->log_u[row] = p.log_u;
          m->lp_old[row] = p.lp_old;
          m->w[row] = p.valid ? p.w : -1;
        }
        return true;
      };
      Prep cur{}, nxt{};
      if (tile0 < ntiles) cur = prep(tile0, false);  // (the old log-prob is state: it is read behind the barrier)
      if (h == 0) {
        // everything above (barrier set-up, factor copy, first draws and index lookups) overlapped the tail of
        // the previous kernel when this one was launched as its programmatic dependent; the state that
        // kernel wrote may be read from here on
        pdl_wait();
        pdl_launch_dependents();
        // (a completed predecessor kernel needs no proxy fence: griddepcontrol.wait returns with its writes
        // performed; the fence costs ~1 us per launch).  Sharded: the peer barrier is NOT taken here -- tiles
        // whose partners are local start at once; issue() takes it before the first remote fetch, pair 0's
        // producer right after its first tile at the latest, the consumers before their first store.
        if (multi && !a.aperm && !peers_ready()) return;  // natural tile order: barrier first, as before
        // launch start: get the first rows moving before anything else.  All 8 pairs asking at once is a
        // 19 MB burst (148 SMs x 8 slots x 16 KB) during which nobody computes -- and, sharded, a burst on
        // the NVLink ports; with the stagger the second pair of each sub-partition asks only when the first
        // pair's rows are in, so one consumer per sub-partition starts after half the burst.
        if (tile0 < ntiles) {
          // (best effort: a bounded peek at the neighbour's barrier, never a dependency)
          if (a.dmma_stagger && pair >= DMMA_CONSUMERS / 2)
            mbar_wait_for(barFull + pair - DMMA_CONSUMERS / 2, 0, multi ? 40000 : 12000);
          if (tlp) tlp[6] = clock64() - t_entry_p;
          if (!issue(cur, (int)(k & 1u), true)) return;
        }
        // pair 0 takes the barrier now if its first tile did not need it (the flags normally arrive while that
        // tile's rows are in flight); the other producers only wait for it inside issue(), when they need it
        if (pair == 0 && !peers_ready()) return;
        if (tile0 + tstride < ntiles) nxt = prep(tile0 + tstride, true);
      } else {
        if (tile0 + tstride < ntiles) nxt = prep(tile0 + tstride, false);
        // every CTA (of every rank) has finished writing half-step h-1: the state may be read again
        bool ok = true;
        if (lane == 0) ok = grid_wait(gbar, gbar_base + (unsigned long long)h * gridDim.x, a.status);
        ok = __shfl_sync(0xffffffffu, ok, 0);
        if (!ok) {
          *sAbort = 1;
          return;
        }
        asm volatile("fence.proxy.async;" ::: "memory");  // generic-proxy writes of other SMs -> our TMA reads
        // (persistent launches are single-GPU: the host runs sharded ensembles one half-step per launch)
        if (tile0 < ntiles) {
          // the slot was released by the consumer at the end of the previous half-step's last tile
          if (k > 0 && !mbar_wait_abortable(barFree + pair, (k - 1) & 1u, sAbort)) return;
          if (!issue(cur, (int)(k & 1u), true)) return;
        }
      }
      for (int64_t tile = tile0; tile < ntiles; tile += tstride, ++k) {
        // ---- rows of this tile have landed: form the proposal over the partner rows
        const double zz = __shfl_sync(0xffffffffu, cur.zz, g);
        if (!mbar_wait_abortable(barFull + pair, k & 1u, sAbort)) return;
        long long* tlq = (tlp && h == nhalf - 1 && (tile - tile0) / tstride < TL_TILES && lane == 0)
                             ? tlp + ((tile - tile0) / tstride) * TL_EVENTS : nullptr;
        if (tlq) tlq[7] = clock64() - t_entry_p;
#pragma unroll
        for (int j = 0; j < KB; ++j) {
          const double2 s2 = *reinterpret_cast<const double2*>(myS + 8 * j);
          const double2 c2 = *reinterpret_cast<const double2*>(myC + 8 * j);
          // stretch.py:33  q = c - (c - s) * zz, each op rounded once (no FMA contraction)
          double2 q2;
          q2.x = __dsub_rn(c2.x, __dmul_rn(__dsub_rn(c2.x, s2.x), zz));
          q2.y = __dsub_rn(c2.y, __dmul_rn(__dsub_rn(c2.y, s2.y), zz));
          *reinterpret_cast<double2*>(myC + 8 * j) = q2;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(barReady + pair);
        if (tlq) tlq[8] = clock64() - t_entry_p;
        // ---- as soon as the consumer has the proposal in registers, refill the slot
        if (tile + tstride < ntiles) {
          cur = nxt;
          if (!mbar_wait_abortable(barFree + pair, k & 1u, sAbort)) return;
          if (tlq && (tile - tile0) / tstride + 1 < TL_TILES)
            tlq[TL_EVENTS + 6] = clock64() - t_entry_p;  // (stamp 6 of the NEXT tile: its rows are requested)
          if (!issue(cur, (int)((k + 1) & 1u), h > 0 && tile == tile0)) return;
          if (tile + 2 * tstride < ntiles) nxt = prep(tile + 2 * tstride, true);
        }
      }
    }
    return;
  }

  // ================================ consumer: DMMA, accept, update ================================
  // optional per-tile timestamps of the LAST half-step (cycles since this warp entered the kernel):
  // 1 wait start, 2 proposal ready, 3 proposal in registers, 4 DMMA block done, 5 tile done
  const long long t_entry = clock64();
  long long* tl = a.timeline ? a.timeline + ((size_t)blockIdx.x * DMMA_CONSUMERS + pair) * TL_TILES * TL_EVENTS : nullptr;
  pdl_wait();  // nothing of this warp's global traffic may overtake the previous kernel
  pdl_launch_dependents();
  // On an abort a consumer stops working but keeps walking the same sequence of named barriers as its
  // siblings, so nobody is left waiting for a warp that left.
  bool alive = mbar_wait_abortable(barL, 0, sAbort);
  for (int h = 0; h < nhalf; ++h) {
    const HalfDesc d = (h == 0) ? d0 : descs[h];
    const int2 rg = a.range ? a.range[(size_t)d.order_step * MAX_SPLITS + d.split] : make_int2(0, d.a_count);
    const int64_t ntiles = ((int64_t)rg.y - rg.x + 7) >> 3;
    unsigned kk = 0;
    bool peers_passed = false;
    for (int64_t tile = tile0; alive && tile < ntiles; tile += tstride, ++k, ++kk) {
      const TileMeta* m = meta + (k & 1u);
      long long* tlk = (tl && h == nhalf - 1 && kk < TL_TILES && lane == 0) ? tl + kk * TL_EVENTS : nullptr;
      if (tlk) {
        tlk[0] = (long long)tile;
        tlk[1] = clock64() - t_entry;
      }
      if (!mbar_wait_abortable(barReady + pair, k & 1u, sAbort)) {
        alive = false;
        break;
      }
      if (tlk) tlk[2] = clock64() - t_entry;
      double q[2 * KB];
#pragma unroll
      for (int j = 0; j < KB; ++j) {
        const double2 q2 = *reinterpret_cast<const double2*>(myC + 8 * j);
        q[2 * j + 0] = q2.x;
        q[2 * j + 1] = q2.y;
      }
      const int32_t w = m->w[g];
      const double factor = m->factor[g], log_u = m->log_u[g], lp_old = m->lp_old[g];
      __syncwarp();
      if (lane == 0) mbar_arrive(barFree + pair);  // slot and meta may be refilled while this tile computes
      if (tlk) tlk[3] = clock64() - t_entry;

      // ---- y = L^T (q - mu) block by block on the tensor pipe; rs = sum_n y_n^2
      double rs = 0.0;
      const double* bptr = sL + 2 * lane;  // one 16-byte load feeds the two k-halves of a block pair
#pragma unroll
      for (int nb0 = 0; nb0 < KB; nb0 += NI) {
        double c[NI][2][2];
#pragma unroll
        for (int n = 0; n < NI; ++n) c[n][0][0] = c[n][0][1] = c[n][1][0] = c[n][1][1] = 0.0;
#pragma unroll
        for (int j = nb0; j < KB; ++j) {
          double x0 = q[2 * j + 0], x1 = q[2 * j + 1];
          if (HAS_MEAN) {
            const double2 m2 = *reinterpret_cast<const double2*>(sMu + 8 * j + 2 * t);
            x0 -= m2.x;
            x1 -= m2.y;
          }
#pragma unroll
          for (int n = 0; n < NI; ++n) {
            if (nb0 + n < KB && j >= nb0 + n) {
              const double2 b2 = *reinterpret_cast<const double2*>(bptr);
              dmma884(c[n][0][0], c[n][0][1], x0, b2.x);
              dmma884(c[n][1][0], c[n][1][1], x1, b2.y);
              bptr += 64;
            }
          }
        }
#pragma unroll
        for (int n = 0; n < NI; ++n) {
          const double y0 = c[n][0][0] + c[n][1][0], y1 = c[n][0][1] + c[n][1][1];
          rs = fma(y0, y0, rs);
          rs = fma(y1, y1, rs);
        }
      }
      rs += __shfl_xor_sync(0xffffffffu, rs, 1);
      rs += __shfl_xor_sync(0xffffffffu, rs, 2);
      const double lp_new = -0.5 * rs;
      if (tlk) tlk[4] = clock64() - t_entry;

      // ---- guards (ensemble.py:476-479, 550-551): a non-finite lp is the only way
      // a non-finite coordinate can show, so the element scan is off the fast path
      if (!isfinite(lp_new)) {
        bool any_inf = false, any_nan = false;
#pragma unroll
        for (int e = 0; e < 2 * KB; ++e) {
          any_inf |= isinf(q[e]);
          any_nan |= isnan(q[e]);
        }
        if (any_inf) atomicOr(a.status, FLAG_INF_PARAM);
        if (any_nan) atomicOr(a.status, FLAG_NAN_PARAM);
        if (isnan(lp_new)) atomicOr(a.status, FLAG_NAN_LOGPROB);
      }

      // ---- Metropolis accept + in-place update (red_blue.py:96-104, move.py:29-34)
      const double lnpdiff = __dsub_rn(__dadd_rn(factor, lp_new), lp_old);
      const bool acc = (w >= 0) && (lnpdiff > log_u);
      if (multi && !peers_passed) {
        // sharded: a slower peer may still be reading this rank's rows for ITS previous half-step; nothing is
        // overwritten before every peer has published that it is through (normally true long before now)
        while (*sPeers <= h) {
          if (*sAbort) break;
          __nanosleep(64);
        }
        peers_passed = !*sAbort;
        if (!peers_passed) {
          alive = false;
          break;
        }
      }
      if (acc) {
        double* dst = a.coords + (size_t)w * D + 2 * t;
#pragma unroll
        for (int j = 0; j < KB; ++j) *reinterpret_cast<double2*>(dst + 8 * j) = make_double2(q[2 * j], q[2 * j + 1]);
      }
      if (w >= 0 && t == 0) {
        if (acc) {
          a.logp[w] = lp_new;
          atomicAdd(a.nacc + w, 1ull);  // RED: fire and forget
        }
        a.accepted[w] = acc ? 1 : 0;
      }
      if (tlk) tlk[5] = clock64() - t_entry;
    }
    if (h + 1 < nhalf) {
      // this CTA's updates of half-step h are out: tell the grid (consumer warps only, named barrier 1)
      __threadfence();
      asm volatile("bar.sync 1, %0;" ::"r"(32 * DMMA_CONSUMERS) : "memory");
      if (*sAbort) alive = false;
      if (tid == 0 && alive) {
        __threadfence();
        atomicAdd(gbar, 1ull);
      }
    }
  }
  if (multi) {
    // the last CTA of this rank to finish tells every peer that the launch's last half-step is done here
    // (an aborted CTA does not count: the peers then time out as well and every rank reports the failure)
    __threadfence_system();
    asm volatile("bar.sync 1, %0;" ::"r"(32 * DMMA_CONSUMERS) : "memory");
    if (tid == 0 && !*sAbort) {
      const unsigned prev = atomicAdd(a.p2p_done, 1u);
      if (prev == gridDim.x - 1) {
        *a.p2p_done = 0;  // re-armed for the next launch (stream order: nobody else touches it now)
        __threadfence_system();
        for (int r = 0; r < a.p2p_nranks; ++r)
          if (r != a.p2p_rank)
            atomicExch_system(a.p2p_peer_flags[r] + a.p2p_rank, a.p2p_signal + (unsigned)(nhalf - 1));
      }
    }
  }
}

// ===========================================================================
// stand-alone log-probability of dense-Gaussian rows on the tensor pipe
// (EnsembleSampler.compute_log_prob and the initial state, ensemble.py:350-358,458-553)
// ===========================================================================
template <int KB, bool HAS_MEAN>
__global__ void __launch_bounds__(256) logprob_dense_dmma_kernel(const ModelDev m, const double* __restrict__ x,
                                                                 const int64_t rows, double* __restrict__ out,
                                                                 int* status) {
  constexpr int D = 8 * KB;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sL = reinterpret_cast<double*>(smem_raw);
  double* sMu = sL + (size_t)packed_blocks(KB) * 32;
  uint64_t* barL = reinterpret_cast<uint64_t*>(sMu + D);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  if (tid == 0) {
    mbar_init(barL, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (HAS_MEAN)
    for (int k = tid; k < D; k += blockDim.x) sMu[k] = m.params[k];
  __syncthreads();
  if (tid == 0) {
    constexpr unsigned bytes = (unsigned)((size_t)packed_blocks(KB) * 32 * sizeof(double));
    mbar_arrive_expect_tx(barL, bytes);
    bulk_g2s(sL, m.chol, bytes, barL);
  }
  const int64_t ntiles = (rows + 7) >> 3;
  bool waited = false;
  for (int64_t tile = (int64_t)blockIdx.x * 8 + warp; tile < ntiles; tile += (int64_t)gridDim.x * 8) {
    int64_t r = tile * 8 + g;
    const bool valid = r < rows;
    if (!valid) r = rows - 1;
    const double* src = x + (size_t)r * D + 2 * t;
    double q[2 * KB];
    bool any_inf = false, any_nan = false;
#pragma unroll
    for (int j = 0; j < KB; ++j) {
      const double2 v = __ldcg(reinterpret_cast<const double2*>(src + 8 * j));
      q[2 * j + 0] = v.x;
      q[2 * j + 1] = v.y;
      any_inf |= isinf(v.x) | isinf(v.y);
      any_nan |= isnan(v.x) | isnan(v.y);
    }
    if (valid && any_inf) atomicOr(status, FLAG_INF_PARAM);  // ensemble.py:476-477
    if (valid && any_nan) atomicOr(status, FLAG_NAN_PARAM);  // ensemble.py:478-479
    if (!waited) {
      mbar_wait(barL, 0);
      waited = true;
    }
    double rs = tile_sumsq<KB, HAS_MEAN>(q, sL, sMu, lane, t);
    rs += __shfl_xor_sync(0xffffffffu, rs, 1);
    rs += __shfl_xor_sync(0xffffffffu, rs, 2);
    const double lp = -0.5 * rs;
    if (valid && t == 0) {
      out[r] = lp;
      if (isnan(lp)) atomicOr(status, FLAG_NAN_LOGPROB);  // ensemble.py:550-551
    }
  }
}

template <int KB>
cudaError_t launch_lp_t(const ModelDev& m, const double* x, int64_t rows, double* out, int* status, int max_grid,
                        cudaStream_t st) {
  const size_t smem = ((size_t)packed_blocks(KB) * 32 + 8 * KB) * sizeof(double) + sizeof(uint64_t);
  const bool has_mean = m.s0 != 0.0;
  auto kern = has_mean ? logprob_dense_dmma_kernel<KB, true> : logprob_dense_dmma_kernel<KB, false>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  if (rows <= 0) return cudaSuccess;
  const int64_t want = (((rows + 7) >> 3) + 7) / 8;
  const int grid = (int)(want < max_grid ? want : max_grid);
  kern<<<grid, 256, smem, st>>>(m, x, rows, out, status);
  return cudaGetLastError();
}

template <int KB>
cudaError_t launch_t(const HalfStepArgs& a, const HalfDesc& d0, const HalfDesc* descs_dev, int nhalf, int max_count,
                     unsigned long long* gbar, unsigned long long gbar_base, int max_grid, bool pdl,
                     LaunchShape* shape, cudaStream_t st) {
  const size_t smem = SmemLayout<KB>::total_bytes;
  const bool has_mean = a.model.s0 != 0.0;  // set by eb_model_set when mu != 0
  auto kern = has_mean ? half_step_dense_dmma_kernel<KB, true> : half_step_dense_dmma_kernel<KB, false>;
  // the opt-in to > 48 KB of dynamic shared memory is per device: remember where it has been done
  static bool configured[2][64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !configured[has_mean][dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) configured[has_mean][dev] = true;
  }
  const int64_t ntiles = max_count > 0 ? ((int64_t)max_count + 7) / 8 : 0;
  const int grid = (int)(ntiles < max_grid ? ntiles : max_grid);
  *shape = LaunchShape{SHAPE_DENSE_DMMA, 8, 0, 0, DMMA_CONSUMERS, DMMA_THREADS, nhalf > 0 ? grid : 0, ntiles};
  if (max_count <= 0 || nhalf <= 0) return cudaSuccess;
  HalfStepArgs args = a;
  HalfDesc first = d0;
  if (nhalf == 1) {
    // no grid barrier inside: a plain launch (cooperative launches cost ~2 us more each).  With `pdl`
    // the kernel is a programmatic dependent of the previous kernel in the stream: its prologue
    // (barrier set-up, factor copy, first draws, L2 prefetch of its own rows) overlaps that kernel's tail.
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(DMMA_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, args, first, descs_dev, nhalf, gbar, gbar_base);
  }
  // cooperative launch: the grid barrier between half-steps needs every CTA resident
  void* params[] = {(void*)&args, (void*)&first, (void*)&descs_dev, (void*)&nhalf, (void*)&gbar, (void*)&gbar_base};
  return cudaLaunchCooperativeKernel((const void*)kern, dim3(grid), dim3(DMMA_THREADS), params, smem, st);
}

}  // namespace

// any ndim that is a multiple of 8 up to 128 (the proposal tile lives in D/4 registers per lane)
bool dense_dmma_supported(int D) { return D >= 8 && D <= 128 && D % 8 == 0; }

size_t dense_dmma_factor_doubles(int D) { return (size_t)packed_blocks(D / 8) * 32; }

// L: row-major lower-triangular factor (A = L L^T).  Packed in the order the
// kernel consumes it: for each group of NI 8-column tiles, for each 8-row group
// j, for each tile nb of the group with j >= nb, the two 4x8 fragments (half = 0, 1)
// interleaved per lane: lane (g, t) holds L[8j + 2t + half][8nb + g], half = 0, 1 side by side.
void dense_dmma_pack_factor(const double* L, int D, double* packed) {
  const int KB = D / 8;
  size_t idx = 0;
  for (int nb0 = 0; nb0 < KB; nb0 += NI)
    for (int j = nb0; j < KB; ++j)
      for (int n = 0; n < NI; ++n) {
        const int nb = nb0 + n;
        if (nb >= KB || j < nb) continue;
        for (int lane = 0; lane < 32; ++lane)
          for (int half = 0; half < 2; ++half) {  // the two k-halves of a lane sit side by side (one LDS.128)
            const int g = lane >> 2, t = lane & 3;
            packed[idx++] = L[(size_t)(8 * j + 2 * t + half) * D + (8 * nb + g)];
          }
      }
}

cudaError_t launch_logprob_dense_dmma(const ModelDev& m, int D, const double* x, int64_t rows, double* out,
                                      int* status, int max_grid, cudaStream_t st) {
#define EB_LP_CASE(KB) \
  case 8 * KB:         \
    return launch_lp_t<KB>(m, x, rows, out, status, max_grid, st);
  switch (D) {
    EB_LP_CASE(1)
    EB_LP_CASE(2)
    EB_LP_CASE(3)
    EB_LP_CASE(4)
    EB_LP_CASE(5)
    EB_LP_CASE(6)
    EB_LP_CASE(7)
    EB_LP_CASE(8)
    EB_LP_CASE(9)
    EB_LP_CASE(10)
    EB_LP_CASE(11)
    EB_LP_CASE(12)
    EB_LP_CASE(13)
    EB_LP_CASE(14)
    EB_LP_CASE(15)
    EB_LP_CASE(16)
  }
#undef EB_LP_CASE
  return cudaErrorNotSupported;
}

cudaError_t launch_dense_dmma(const HalfStepArgs& a, const HalfDesc& d0, const HalfDesc* descs_dev, int nhalf,
                              int max_count, unsigned long long* gbar, unsigned long long gbar_base, int max_grid,
                              bool pdl, LaunchShape* shape, cudaStream_t st) {
#define EB_DMMA_CASE(KB) \
  case 8 * KB:           \
    return launch_t<KB>(a, d0, descs_dev, nhalf, max_count, gbar, gbar_base, max_grid, pdl, shape, st);
  switch (a.D) {
    EB_DMMA_CASE(1)
    EB_DMMA_CASE(2)
    EB_DMMA_CASE(3)
    EB_DMMA_CASE(4)
    EB_DMMA_CASE(5)
    EB_DMMA_CASE(6)
    EB_DMMA_CASE(7)
    EB_DMMA_CASE(8)
    EB_DMMA_CASE(9)
    EB_DMMA_CASE(10)
    EB_DMMA_CASE(11)
    EB_DMMA_CASE(12)
    EB_DMMA_CASE(13)
    EB_DMMA_CASE(14)
    EB_DMMA_CASE(15)
    EB_DMMA_CASE(16)
  }
#undef EB_DMMA_CASE
  return cudaErrorNotSupported;
}

}  // namespace eb
