// pma.cu -- K4: PMA.train()/test() (Dyna-Q with Mattar & Daw prioritized memory access:
// replay of the backup with the largest gain x need) for N independent agents.
//
// Reference: agent/pma.py:167-353 (trial loop, online n-step update_q) and
// memory/pma.py:104-496 (store, replay, compute_gain_batch, compute_gain, compute_need,
// update_sr, update_q).  Semantics: SURVEY.md Appendix A.7.
//
// Kernels (cobel_pma_run picks the path, see run<A>()):
//
//   pma_main_kernel  ONE WARP PER AGENT.  reset + start-of-trial replay + the online steps [+ update_sr +
//                    end-of-trial replay].  Q, M.rewards, M.states|terminals, the utility vector and the need
//                    row live in shared memory (14 KB per agent at 10x10, 16 agents per SM); T stays in HBM
//                    (one row read+written per step).  Replay: the gain of every one-step backup depends on two
//                    Q rows, so after the first iteration of a replay call only the backups whose rows were
//                    touched by the previous update are re-evaluated (compacted to one lane-parallel pass) --
//                    bit-identical to the reference's full recomputation; gain x need x mask, the exact-tie
//                    arg-max draw and the n-step update are warp passes with shuffle reductions (no block
//                    barriers).
//   update_sr, banded (CobelPMAParams.sr_band >= 0): replay reads ONE row of SR per call, and T of a W-wide
//                    gridworld has half bandwidth W: pma_band_factor_kernel / pma_band_solve_kernel, ONE WARP PER
//                    AGENT between the main kernel's launches, factorise the band of I - gamma T (or run the
//                    banded GTH elimination for the stationary need of timed-out trials) and solve for the rows
//                    the replays need; SR is refreshed once per call by pma_sr_band_kernel from the last factors.
//   update_sr, dense (any T): pma_sr_kernel, ONE CTA PER AGENT, after every trial (the main kernel is then
//                    launched once per trial, per-agent state carried in HBM): SR = inv(I - gamma T) by
//                    register-tiled Gauss-Jordan (no pivoting: I - gamma T is strictly diagonally dominant); for
//                    agents whose trial timed out also the stationary distribution (the reference's LAPACK
//                    dgeev `need`) by the subtraction-free GTH elimination.
//   With replays on, the main kernel is launched per phase (MainPhase): update_sr sits between a trial's steps
//   and its end replay, and the per-agent state travels in `carry`.
//   cobel_pma_replay (the stand-alone PMAMemory.replay, replay_only<A>) runs the end-replay phase alone: after the
//   dense update_sr kernel up to 160 states and 1024 backups, after the banded kernels beyond
//   (pma_band_stationary_kernel when only the stationary need is wanted).
//
// (v1 ran everything in one CTA per agent and was barrier-bound: 7 of 8 warps waited for warp 0
//  through ~12 block barriers per replay iteration, profiles/r1_pma_v1_cta_per_agent.txt.)
// The main kernel is instruction-fetch bound (its replay loop is as large as the L1.5 instruction cache): the
// rarely executed routines are __noinline__, runtime loops are not unrolled, fp64 division and the Philox refill
// are single shared copies (DESIGN.md K4).
//
// Exactness: everything except SR / the stationary vector follows the reference's operation
// order bit for bit; those two come from a different (but 1e-13-accurate) factorisation than
// LAPACK's, which only matters if two distinct utilities are closer than that -- the smallest
// relative gap seen is reported per agent (`min_gap`) as a certificate.
#include "warp_agent.cuh"
#include "tma.cuh"

namespace {

constexpr int kThreads = 256;        // pma_sr_kernel: 16 x 16 thread grid for the register-tiled eliminations
constexpr int kMainWarps = 4;        // pma_main_kernel: agents (warps) per CTA
constexpr int kMaxSeq = 64;          // longest n-step sequence (replay batch) supported

// Policy probabilities for one Q row (thread-local): policy/greedy.py:60-88,117-147, policy/softmax.py:60-88.
// qpar[n-1] = par/n and qom[n-1] = (1-par)/n are the cached quotients.
// The PMA kernels are instruction-fetch bound (their replay loop alone exceeds the 32 KB L1.5 instruction cache):
// the fp64 division (a ~40-instruction sequence) is one shared copy here.
__device__ __noinline__ double pdiv(double a, double b) { return __ddiv_rn(a, b); }

// t[idx] by a select chain: a dynamically indexed register array would live in local memory
template <int A>
COBEL_DEV double pick(const double (&t)[A], int idx) {
  double v = t[0];
#pragma unroll
  for (int a = 1; a < A; ++a) v = idx == a ? t[a] : v;
  return v;
}

template <int A>
COBEL_DEV void probs_row(const double (&v)[A], uint32_t mask, int kind, double par, const double (&qpar)[A], const double (&qom)[A],
                         double (&p)[A]) {
  double m = -__longlong_as_double(0x7FF0000000000000ll);
#pragma unroll
  for (int a = 0; a < A; ++a) m = (mask >> a & 1u) ? xmax(m, v[a]) : m;
  const int nv = __popc(mask);
  if (kind == COBEL_POLICY_SOFTMAX) {
    double sum = 0.0;
#pragma unroll
    for (int a = 0; a < A; ++a) {
      p[a] = 0.0;
      if (mask >> a & 1u) { p[a] = exp(xmul(xsub(v[a], m), par)); sum = xadd(sum, p[a]); }
    }
    if (A == 8 && nv == 8) sum = np_sum<A>(p);             // np.sum over exactly 8 values is a tree, not a loop
#pragma unroll
    for (int a = 0; a < A; ++a)
      if (mask >> a & 1u) p[a] = pdiv(p[a], sum);
    return;
  }
  uint32_t ties = 0;
#pragma unroll
  for (int a = 0; a < A; ++a) ties |= (v[a] == m ? 1u : 0u) << a;
  ties &= mask;
  const int k = __popc(ties);
  const double tie = pick<A>(qom, k - 1);
  double top, low;
  if (kind == COBEL_POLICY_EPS_GREEDY) {
    const double base = pick<A>(qpar, nv - 1);
    top = xadd(base, tie); low = xadd(base, 0.0);
  } else {
    const int d = nv - k > 1 ? nv - k : 1;
    top = xadd(tie, 0.0); low = xadd(0.0, pick<A>(qpar, d - 1));
  }
#pragma unroll
  for (int a = 0; a < A; ++a) p[a] = (mask >> a & 1u) ? ((ties >> a & 1u) ? top : low) : 0.0;
}

template <int A>
COBEL_DEV double sum_seq(const double (&x)[A]) { return np_sum<A>(x); }    // np.sum over one row of A values

// ---------------------------------------------------------------------------
// Register-tiled dense eliminations on an S x S matrix distributed over the 16 x 16 thread
// grid of the CTA: thread (ty, tx) owns elements (ty + 16 r, tx + 16 c), r, c < TILE.  Each
// elimination step broadcasts one pivot row and one pivot column through shared memory
// (double-buffered: one barrier per step) and updates the tiles with TILE*TILE DFMAs per
// thread, i.e. the S^3 work runs out of registers at the fp64 pipe rate instead of the
// shared-memory rate.  These two routines are the only non-bit-exact arithmetic of the kernel
// (the reference calls LAPACK here), so FMA contraction is used deliberately.
// ---------------------------------------------------------------------------
template <int TILE>
struct Tile {
  double m[TILE][TILE];
};

// SR = inv(I - gamma T) by in-place Gauss-Jordan without pivoting (I - gamma T is strictly
// diagonally dominant, so any pivot order is stable; pivots are taken in the order
// k = ty0 + 16 r0 with r0 as the unrolled outer loop, which makes the pivot row / column of a
// thread's tile a compile-time register index).  The pivot row / column need no special-casing
// in the update: the owner of the pivot publishes piv + 1 in the row slot and piv - 1 in the
// column slot, so that the generic m -= f_i * (rowk_j / piv) also yields the scaled pivot row,
// -f_i / piv in the pivot column and 1 / piv on the pivot (cancellation error ~ eps * piv).
template <int TILE>
__device__ __forceinline__ void gauss_jordan_inverse(const double* __restrict__ Tg, double gsr, double* SRg, int S,
                                                     double* buf, int tid, int& flags) {
  const int ty = tid >> 4, tx = tid & 15;
  constexpr int SP = TILE * 16 + 2;                 // row / column slots + {piv, 1/piv}
  Tile<TILE> t;
#pragma unroll
  for (int r = 0; r < TILE; ++r)
#pragma unroll
    for (int c = 0; c < TILE; ++c) {
      const int i = ty + 16 * r, j = tx + 16 * c;
      double v = i == j ? 1.0 : 0.0;
      if (i < S && j < S) v -= gsr * Tg[(size_t)i * S + j];
      t.m[r][c] = v;
    }
#pragma unroll
  for (int r0 = 0; r0 < TILE; ++r0) {
    for (int ty0 = 0; ty0 < 16; ++ty0) {
      const int k = ty0 + 16 * r0;
      if (k >= S) break;
      double* rowk = buf + (k & 1) * 2 * SP;
      double* colk = rowk + SP;
      if (ty == ty0) {
#pragma unroll
        for (int c = 0; c < TILE; ++c) rowk[tx + 16 * c] = t.m[r0][c];
      }
      if (tx == ty0) {
#pragma unroll
        for (int r = 0; r < TILE; ++r) colk[ty + 16 * r] = t.m[r][r0];
        if (ty == ty0) {                              // owner of the pivot
          const double piv = t.m[r0][r0];
          if (!(fabs(piv) > 1e-300)) flags |= COBEL_FLAG_SINGULAR;
          rowk[k] = piv + 1.0;
          colk[k] = piv - 1.0;
          rowk[SP - 1] = 1.0 / piv;
        }
      }
      __syncthreads();
      const double ipiv = rowk[SP - 1];
      double rk[TILE];
#pragma unroll
      for (int c = 0; c < TILE; ++c) rk[c] = rowk[tx + 16 * c] * ipiv;
#pragma unroll
      for (int r = 0; r < TILE; ++r) {
        const double f = colk[ty + 16 * r];
#pragma unroll
        for (int c = 0; c < TILE; ++c) t.m[r][c] = fma(-f, rk[c], t.m[r][c]);
      }
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < TILE; ++r)
#pragma unroll
    for (int c = 0; c < TILE; ++c) {
      const int i = ty + 16 * r, j = tx + 16 * c;
      if (i < S && j < S) SRg[(size_t)i * S + j] = t.m[r][c];
    }
  __syncthreads();
}

// Stationary distribution of the row-stochastic T by GTH (Grassmann-Taksar-Heyman) elimination,
// returned in x[0..S) scaled to unit 2-norm.  Mat receives the eliminated matrix (scratch).
// States are eliminated in descending order k = S-1 .. 1 (r0 unrolled as above).
template <int TILE>
__device__ __forceinline__ void gth_stationary(const double* __restrict__ Tg, double* Mat, double* x, int S, double* buf,
                                               int tid, int& flags) {
  const int ty = tid >> 4, tx = tid & 15, lane = tid & 31;
  constexpr int SP = TILE * 16 + 2;
  Tile<TILE> t;
#pragma unroll
  for (int r = 0; r < TILE; ++r)
#pragma unroll
    for (int c = 0; c < TILE; ++c) {
      const int i = ty + 16 * r, j = tx + 16 * c;
      t.m[r][c] = (i < S && j < S) ? Tg[(size_t)i * S + j] : 0.0;
    }
#pragma unroll
  for (int r0 = TILE - 1; r0 >= 0; --r0) {
    for (int ty0 = 15; ty0 >= 0; --ty0) {
      const int k = ty0 + 16 * r0;
      if (k >= S || k < 1) continue;
      double* rowk = buf + (k & 1) * 2 * SP;
      double* colk = rowk + SP;
      if (ty == ty0) {
#pragma unroll
        for (int c = 0; c < TILE; ++c) rowk[tx + 16 * c] = t.m[r0][c];
      }
      if (tx == ty0) {
#pragma unroll
        for (int r = 0; r < TILE; ++r) colk[ty + 16 * r] = t.m[r][r0];
      }
      __syncthreads();
      // every warp forms s = sum_{j<k} P[k][j] with the same reduction tree
      double ssum = 0.0;
      for (int j = lane; j < k; j += 32) ssum += rowk[j];
      for (int d = 16; d > 0; d >>= 1) ssum += shfl_f64_xor(ssum, d);
      if (!(ssum > 0.0)) { flags |= COBEL_FLAG_SINGULAR; ssum = 1.0; }
      const double inv = 1.0 / ssum;
      // only rows / columns below k take part: with k = ty0 + 16 r0 these are the tile rows and
      // columns 0..r0, a compile-time bound -- the work shrinks with k (S^3/3 instead of S^3)
      double rk[TILE];
#pragma unroll
      for (int c = 0; c < TILE; ++c) {
        if (c <= r0) { const int j = tx + 16 * c; rk[c] = j < k ? rowk[j] : 0.0; }
      }
#pragma unroll
      for (int r = 0; r < TILE; ++r) {
        if (r <= r0) {
          const int i = ty + 16 * r;
          const double f = i < k ? colk[i] * inv : 0.0;
#pragma unroll
          for (int c = 0; c < TILE; ++c)
            if (c <= r0) t.m[r][c] = fma(f, rk[c], t.m[r][c]);
          // column k keeps the scaled entries P[i][k] / s for the back-substitution
          if (tx == ty0 && i < k) t.m[r][r0] = f;
        }
      }
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < TILE; ++r)
#pragma unroll
    for (int c = 0; c < TILE; ++c) {
      const int i = ty + 16 * r, j = tx + 16 * c;
      if (i < S && j < S) Mat[j * S + i] = t.m[r][c];      // transposed: column k becomes a contiguous row
    }
  __syncthreads();
  if (tid < 32) {                                   // x_0 = 1, x_k = sum_{i<k} x_i P[i][k]: one warp, no block barriers
    if (lane == 0) x[0] = 1.0;
    __syncwarp();
    for (int k = 1; k < S; ++k) {
      double acc = 0.0;
      for (int i = lane; i < k; i += 32) acc = fma(x[i], Mat[k * S + i], acc);
      for (int d = 16; d > 0; d >>= 1) acc += shfl_f64_xor(acc, d);
      if (lane == 0) x[k] = acc;
      __syncwarp();
    }
    double sq = 0.0;
    for (int i = lane; i < S; i += 32) sq = fma(x[i], x[i], sq);
    for (int d = 16; d > 0; d >>= 1) sq += shfl_f64_xor(sq, d);
    const double nrm = sqrt(sq);
    for (int i = lane; i < S; i += 32) x[i] = fabs(x[i]) / nrm;
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------
// pma_sr_kernel: one CTA per agent.  SR <- inv(I - gamma T); if the agent's last trial timed
// out (carry[.,0] < 0) also the stationary `need` vector into need_scratch[n].
// ---------------------------------------------------------------------------
template <int TILE>
__global__ void __launch_bounds__(kThreads, TILE <= 7 ? 2 : 1) pma_sr_kernel(const __grid_constant__ CobelPMAParams p,
                                                                            const int final_only) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, tid = threadIdx.x;
  const int64_t n = blockIdx.x;
  double* elim = reinterpret_cast<double*>(smem);                 // 2 x (pivot row + pivot column)
  double* xv = elim + 4 * (TILE * 16 + 2);                        // [S] stationary vector
  double* Mat = xv + ((S + 1) & ~1);                              // [S*S] GTH scratch
  int flags = 0;
  const double* Tg = p.T + (size_t)n * S * S;
  if (final_only != 2) gauss_jordan_inverse<TILE>(Tg, p.gamma_sr[n], p.SR + (size_t)n * S * S, S, elim, tid, flags);
  if (final_only == 1) {
    // end of a banded call (sr_band >= 0): SR is refreshed once, and the caller's band guarantee is verified
    const int bw = p.sr_band;
    for (int e = tid; e < S * S; e += kThreads) {
      const int i = e / S, j = e - i * S;
      if (abs(i - j) > bw && Tg[e] != 0.0) flags |= COBEL_FLAG_BAND_VIOLATION;
    }
  } else if (p.carry[n * 8 + 0] < 0) {               // (final_only == 2: the stationary need only, SR is left alone)
    gth_stationary<TILE>(Tg, Mat, xv, S, elim, tid, flags);
    for (int e = tid; e < S; e += kThreads) p.need_scratch[(size_t)n * S + e] = xv[e];
  }
  __shared__ int block_flags;                        // the OR of the threads' COBEL_FLAG_* bits (__syncthreads_or gives 0 / 1)
  if (tid == 0) block_flags = 0;
  __syncthreads();
  if (flags) atomicOr(&block_flags, flags);
  __syncthreads();
  if (tid == 0 && block_flags && p.trace.flags) p.trace.flags[n] |= block_flags;
}

// ---------------------------------------------------------------------------
// Banded update_sr (CobelPMAParams.sr_band): replay reads ONE row of SR = inv(M), M = I - gamma T
// (memory/pma.py:401-411), and T of a W-wide gridworld has half bandwidth bw = W, so instead of the S^3 dense
// inverse the band is factorised (S * bw^2 operations, no pivoting: M is strictly diagonally dominant, the
// factors stay inside the band) and x^T M = e_c^T is solved for the row (2 * S * bw).  The result is what the
// dense elimination gives with the multiplications by the exact zeros outside the band left out.
// Band storage in global scratch: b[i * W + (j - i + bw)] = M[i][j], W = 2 bw + 1.
// ---------------------------------------------------------------------------

// 1 / x to ~1 ulp without the IEEE division's slow path: MUFU.RCP64H seed + two Newton steps.  Only the banded
// eliminations use it (not bit-exact by design); their pivots and row sums are far from the subnormal range, and
// anything below 1e-300 raises COBEL_FLAG_SINGULAR first.
COBEL_DEV double fast_rcp(double x) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  y = fma(fma(-x, y, 1.0), y, y);
  y = fma(fma(-x, y, 1.0), y, y);
  return y;
}

COBEL_DEV void cp_async8(double* smem_dst, const double* gsrc, bool valid) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int sz = valid ? 8 : 0;                       // src-size 0: the 8 bytes are zero-filled
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(sa), "l"(gsrc), "r"(sz) : "memory");
}
COBEL_DEV void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
COBEL_DEV void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// The eliminations are latency-critical (S dependent steps), so rows are STREAMED through a small shared-memory
// ring with cp.async kBandAhead rows ahead of the step that needs them: the HBM/L2 latency of T is off the
// dependency chain, and a finished row goes to the global scratch with a fire-and-forget store.
constexpr int kBandAhead = 4;
// rows of the ring: the bw + 1 active rows, one being replaced and kBandAhead in flight, rounded up to a power of two
__host__ __device__ inline int band_ring_rows(int bw) {
  int r = 1;
  while (r < bw + 2 + kBandAhead) r <<= 1;
  return r;
}

struct BandRing {
  double* ring;      // [R][W + 1] shared memory, row i lives in slot i % R (R a power of two).  The pitch W + 1 is even, so
                     // the elements (row k + ii, column k + jj) that the lanes ii of an elimination step touch lie an odd
                     // number of doubles apart: conflict-free
  int S, bw, W, R, lane;
  COBEL_DEV BandRing(double* r, int S_, int bw_, int lane_) : ring(r), S(S_), bw(bw_), W(2 * bw_ + 1), R(band_ring_rows(bw_)), lane(lane_) {}
  COBEL_DEV double* row(int i) const { return ring + (i & (R - 1)) * (W + 1); }
  // one commit group per call, also for rows outside [0, S) (keeps the group arithmetic uniform)
  COBEL_DEV void fetch_T(const double* __restrict__ Tg, int i) const {     // band of row i of the dense T
    if (i >= 0 && i < S)
#pragma unroll 1
      for (int d = lane; d < W; d += 32) {
        const int j = i - bw + d;
        const bool ok = j >= 0 && j < S;
        cp_async8(row(i) + d, Tg + (size_t)i * S + (ok ? j : i), ok);
      }
    cp_async_commit();
  }
  COBEL_DEV void store_band(double* b, int i) const {
#pragma unroll 1
    for (int d = lane; d < W; d += 32) b[(size_t)i * W + d] = row(i)[d];
  }
};

// Factors of M = I - g T into fac (band storage): the diagonal receives 1 / pivot, the sub-diagonal part the
// multipliers.  LU without pivoting.
__device__ __noinline__ int band_lu(const double* __restrict__ Tg, double g, double* fac, double* ringmem, int S, int bw,
                                    int lane) {
  int flags = 0;
  const BandRing rg(ringmem, S, bw, lane);
  const int W = rg.W;
  auto to_M = [&](int i) {                            // T band row -> M band row, in place
    if (i < S) {
#pragma unroll 1
      for (int d = lane; d < W; d += 32) { double* e = rg.row(i) + d; *e = (d == bw ? 1.0 : 0.0) - g * *e; }
    }
  };
#pragma unroll 1
  for (int i = 0; i < bw; ++i) rg.fetch_T(Tg, i);
  cp_async_wait<0>();
  __syncwarp();
#pragma unroll 1
  for (int i = 0; i < bw; ++i) to_M(i);
#pragma unroll 1
  for (int i = bw; i <= bw + kBandAhead; ++i) rg.fetch_T(Tg, i);
#pragma unroll 1
  for (int k = 0; k < S; ++k) {
    cp_async_wait<kBandAhead>();                      // row k + bw has landed
    __syncwarp();
    to_M(k + bw);
    __syncwarp();
    const int nb = min(bw, S - 1 - k);
    double* rk = rg.row(k);
    const double piv = rk[bw];
    if (!(fabs(piv) > 1e-300)) flags |= COBEL_FLAG_SINGULAR;
    const double ipiv = fast_rcp(piv);
    // lane ii = row k + ii of the bw x bw update block: its multiplier, then its bw elements in sequence (the pivot
    // row is a broadcast read).  A flattened (ii, jj) -> lane mapping keeps all 32 lanes busy but spends 24
    // instructions of index arithmetic per element round: 96 per step against 45 here.
    if (lane >= 1 && lane <= nb) {
      double* ri = rg.row(k + lane) + (bw - lane);    // &M[k + ii][k]
      const double* u = rk + bw;                      // &M[k][k]
      const double l = ri[0] * ipiv;
      ri[0] = l;
#pragma unroll 2
      for (int jj = 1; jj <= nb; ++jj) ri[jj] = fma(-l, u[jj], ri[jj]);
    }
    __syncwarp();
    if (lane == 0) rk[bw] = ipiv;
    __syncwarp();
    rg.store_band(fac, k);
    __syncwarp();
    rg.fetch_T(Tg, k + bw + kBandAhead + 1);          // into the slot row k just left
  }
  cp_async_wait<0>();
  __syncwarp();
  return flags;
}

// x = row c of inv(M) from the factors: U^T y = e_c (forward, column sweeps), then L^T x = y (backward, in place).
// x lives in shared memory, `w` (shared scratch of S doubles) holds the right-hand side of the forward sweep; each
// step reads one factor row straight from the global scratch, the loads running four steps ahead of the recurrence.
__device__ __forceinline__ void band_solve_row(const double* fac, double* w, int S, int bw, int c, double* x, int lane) {
  const int W = 2 * bw + 1;
#pragma unroll 1
  for (int e = lane; e < S; e += 32) { w[e] = e == c ? 1.0 : 0.0; x[e] = 0.0; }
  __syncwarp();
  double dg[4], ov[4];                                // 1 / U[j][j] and this lane's off-diagonal entry of row j
  auto diag = [&](int j) -> double { return (j >= 0 && j < S) ? fac[(size_t)j * W + bw] : 0.0; };
  auto upper = [&](int j) -> double { return (j >= 0 && j < S && lane < bw) ? fac[(size_t)j * W + bw + 1 + lane] : 0.0; };
  auto lower = [&](int j) -> double { return (j >= 0 && j < S && lane < bw) ? fac[(size_t)j * W + bw - 1 - lane] : 0.0; };
#pragma unroll
  for (int u = 0; u < 4; ++u) { dg[u] = diag(c + u); ov[u] = upper(c + u); }
#pragma unroll 1
  for (int j0 = c; j0 < S; j0 += 4) {                 // y_j = rhs_j / U[j][j]; rhs_i -= U[j][i] y_j, i in (j, j+bw]
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = j0 + u;
      if (j < S) {
        const double yj = w[j] * dg[u];
        const int nb = min(bw, S - 1 - j);
        if (lane == 0) x[j] = yj;
        if (lane < nb) w[j + 1 + lane] = fma(-ov[u], yj, w[j + 1 + lane]);
        __syncwarp();
        dg[u] = diag(j + 4); ov[u] = upper(j + 4);
      }
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) ov[u] = lower(S - 1 - u);
#pragma unroll 1
  for (int j0 = S - 1; j0 > 0; j0 -= 4) {             // x_j final; x_i -= L[j][i] x_j, i in [j-bw, j)
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = j0 - u;
      if (j > 0) {
        const double xj = x[j];
        const int nb = min(bw, j);
        if (lane < nb) x[j - 1 - lane] = fma(-ov[u], xj, x[j - 1 - lane]);
        __syncwarp();
        ov[u] = lower(j - 4);
      }
    }
  }
}


// Stationary distribution of the banded row-stochastic T by GTH elimination (see gth_stationary), scaled to
// unit 2-norm, into x (shared memory).  fac receives the eliminated rows (column k holds P[i][k] / s_k).
__device__ __noinline__ int band_gth(const double* __restrict__ Tg, double* fac, double* ringmem, int S, int bw, double* x,
                                     int lane) {
  int flags = 0;
  const BandRing rg(ringmem, S, bw, lane);
  // elimination k = S-1 .. 1 works on rows k-bw .. k: stream upwards
#pragma unroll 1
  for (int i = S - 1; i >= S - 1 - bw - kBandAhead; --i) rg.fetch_T(Tg, i);
#pragma unroll 1
  for (int k = S - 1; k >= 1; --k) {
    cp_async_wait<kBandAhead>();                      // row k - bw has landed
    __syncwarp();
    const int nb = min(bw, k);                        // states k-nb .. k-1 take part
    const double* rk = rg.row(k);
    double ssum = lane < nb ? rk[bw - 1 - lane] : 0.0;
    for (int d = 16; d > 0; d >>= 1) ssum += shfl_f64_xor(ssum, d);
    if (!(ssum > 0.0)) { flags |= COBEL_FLAG_SINGULAR; ssum = 1.0; }
    const double inv = fast_rcp(ssum);
    if (lane >= 1 && lane <= nb) {                    // lane ii = row i = k - ii: P[i][k - jj] += P[i][k] / s * P[k][k - jj]
      double* ri = rg.row(k - lane) + (bw + lane);    // &P[i][k]
      const double* u = rk + bw;                      // &P[k][k]
      const double f = ri[0] * inv;
#pragma unroll 2
      for (int jj = 1; jj <= nb; ++jj) ri[-jj] = fma(f, u[-jj], ri[-jj]);
      ri[0] = f;                                      // column k keeps P[i][k] / s
    }
    __syncwarp();
    rg.store_band(fac, k);                                         // (only its scaled super-diagonal part is read again)
    __syncwarp();
    rg.fetch_T(Tg, k - bw - kBandAhead - 1);
  }
  rg.store_band(fac, 0);
  cp_async_wait<0>();
  if (lane == 0) x[0] = 1.0;
  __syncwarp();
  // x_k = sum_{i<k} x_i P[i][k] / s_k: the scaled column k sits in rows k-bw .. k-1 of fac
  auto colk = [&](int k) -> double {                  // lane's entry of the scaled column k (0 outside)
    return (k < S && lane < min(bw, k)) ? fac[(size_t)(k - 1 - lane) * rg.W + bw + 1 + lane] : 0.0;
  };
  double c[4];                                        // loads run four steps ahead of the recurrence
#pragma unroll
  for (int u = 0; u < 4; ++u) c[u] = colk(1 + u);
  for (int k0 = 1; k0 < S; k0 += 4) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int k = k0 + u;
      if (k < S) {
        double acc = lane < min(bw, k) ? x[k - 1 - lane] * c[u] : 0.0;
        for (int d = 16; d > 0; d >>= 1) acc += shfl_f64_xor(acc, d);
        if (lane == 0) x[k] = acc;
        __syncwarp();
        c[u] = colk(k + 4);
      }
    }
  }
  double sq = 0.0;
#pragma unroll 1
  for (int i = lane; i < S; i += 32) sq = fma(x[i], x[i], sq);
  for (int d = 16; d > 0; d >>= 1) sq += shfl_f64_xor(sq, d);
  const double nrm = sqrt(sq);
#pragma unroll 1
  for (int i = lane; i < S; i += 32) x[i] = fabs(x[i]) / nrm;
  __syncwarp();
  return flags;
}

// ---------------------------------------------------------------------------
// pma_band_factor_kernel / pma_band_solve_kernel: M.update_sr() at a trial boundary, launched between the phases of
// pma_main_kernel.  Inside the main kernel (16 warps per SM, all of its shared memory taken by the replay tables)
// the eliminations ran at 0.5 instructions / cycle / scheduler and made up 36 % of the PMA run
// (profiles/r2_pma_v5.txt).
//   factor: carry[.,0] < 0 (the trial timed out): GTH elimination of T, the stationary vector -> need_scratch;
//           always: LU of I - gamma T -> band_scratch (diagonal = 1 / pivot, sub-diagonal part = multipliers);
//           carry[.,0] >= 0: row carry[.,0] of the inverse -> need_scratch
//   solve:  one row of the inverse from the stored factors -> need_scratch:
//           row carry[.,0] for the end replay of a trial that reached a terminal state, row carry[.,4] (the next
//           trial's start state) for the start replay
// ---------------------------------------------------------------------------
constexpr int kBandWarps = 8;                         // agents per CTA (kBandWarpsWide when their rings do not fit)
constexpr int kBandWarpsWide = 6;
struct BandSmem {                                     // per warp (agent)
  int ring, x, w, bytes;
  __host__ __device__ BandSmem(int S, int bw) {
    // the right-hand side `w` of a row solve aliases the ring: the ring is dead once the factors are in the scratch
    const int ringb = band_ring_rows(bw) * (2 * bw + 2) * 8, vecb = ((S + 1) & ~1) * 8;
    ring = 0;
    w = 0;
    x = ringb > vecb ? ringb : vecb;
    bytes = (x + vecb + 15) & ~15;
  }
};

// Agents (warps) per CTA of the band kernels: kBandWarps, or kBandWarpsWide when eight rings do not fit in shared
// memory -- from half band 27 on the ring has 64 rows, and eight agents would need up to 288 KB; six fit for every
// sr_band <= 31 and S <= 512 (at most 216 KB).
inline int band_warps(int S, int bw) { return kBandWarps * BandSmem(S, bw).bytes <= kMaxSmem ? kBandWarps : kBandWarpsWide; }

// (A one-thread-per-agent factor kernel -- window of bw + 2 rows lane-interleaved in shared memory, 5.5
//  instructions per element update, 3x fewer instructions per agent -- measured 1.28 ms against 1.0 ms for this one
//  at 16384 agents: 32 KB of window per 16 agents leave 1.75 warps per scheduler on strictly dependent steps.)
template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) pma_band_factor_kernel(const __grid_constant__ CobelPMAParams p,
                                                                         const int solve_start) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, bw = p.sr_band, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n = (int64_t)blockIdx.x * WARPS + warp;
  if (n >= p.n_agents) return;
  const BandSmem so(S, bw);
  unsigned char* blk = smem + (size_t)warp * so.bytes;
  double* ring = reinterpret_cast<double*>(blk + so.ring);
  double* x = reinterpret_cast<double*>(blk + so.x);
  const double* Tg = p.T + (size_t)n * S * S;
  double* fac = p.band_scratch + (size_t)n * S * (2 * bw + 1);
  int flags = 0;
  if (p.carry[n * 8 + 0] < 0) {
    flags |= band_gth(Tg, fac, ring, S, bw, x, lane);
    double* need = p.need_scratch + (size_t)n * S;
#pragma unroll 1
    for (int e = lane; e < S; e += 32) need[e] = x[e];
    __syncwarp();
  }
  flags |= band_lu(Tg, p.gamma_sr[n], fac, ring, S, bw, lane);
  if (p.carry[n * 8 + 0] >= 0) {                        // the trial ended in a terminal state: need = SR[last]
    double* w = reinterpret_cast<double*>(blk + so.w);
    band_solve_row(fac, w, S, bw, (int)p.carry[n * 8 + 0], x, lane);
    double* need = p.need_scratch + (size_t)n * S;
#pragma unroll 1
    for (int e = lane; e < S; e += 32) need[e] = x[e];
  }
  if (solve_start) {
    // a single starting state: the next trial's awake replay needs SR[start], known before the reset draw -- its
    // row goes to the second plane of need_scratch and the end replay, the reset, the start replay and the steps
    // of the next trial run in ONE launch of the main kernel
    double* w = reinterpret_cast<double*>(blk + so.w);
    __syncwarp();
    band_solve_row(fac, w, S, bw, __ldg(p.world.starts), x, lane);
    double* need = p.need_scratch + (size_t)(p.n_agents + n) * S;
#pragma unroll 1
    for (int e = lane; e < S; e += 32) need[e] = x[e];
  }
  flags = __reduce_or_sync(kFull, flags);
  if (lane == 0 && flags && p.trace.flags) p.trace.flags[n] |= flags;
}

template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) pma_band_solve_kernel(const __grid_constant__ CobelPMAParams p, const int which) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, bw = p.sr_band, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n = (int64_t)blockIdx.x * WARPS + warp;
  if (n >= p.n_agents) return;
  const int64_t c = p.carry[n * 8 + which];          // which = 0: the last state of the trial, 4: the next start state
  if (c < 0) return;                                  // timed-out trial: need_scratch holds the stationary need
  const BandSmem so(S, bw);
  unsigned char* blk = smem + (size_t)warp * so.bytes;
  double* x = reinterpret_cast<double*>(blk + so.x);
  double* w = reinterpret_cast<double*>(blk + so.w);
  band_solve_row(p.band_scratch + (size_t)n * S * (2 * bw + 1), w, S, bw, (int)c, x, lane);
  double* need = p.need_scratch + (size_t)n * S;
#pragma unroll 1
  for (int e = lane; e < S; e += 32) need[e] = x[e];
}

// The factor pass of a stand-alone replay without update_sr: only the agents whose current state is None
// (carry[.,0] < 0) need anything, the stationary vector of the banded GTH -> need_scratch; the others read the stored
// SR row.  (A kernel of its own rather than a mode of pma_band_factor_kernel keeps train()'s instantiations as they are.)
template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) pma_band_stationary_kernel(const __grid_constant__ CobelPMAParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, bw = p.sr_band, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n = (int64_t)blockIdx.x * WARPS + warp;
  if (n >= p.n_agents || p.carry[n * 8 + 0] >= 0) return;
  const BandSmem so(S, bw);
  unsigned char* blk = smem + (size_t)warp * so.bytes;
  double* x = reinterpret_cast<double*>(blk + so.x);
  int flags = band_gth(p.T + (size_t)n * S * S, p.band_scratch + (size_t)n * S * (2 * bw + 1),
                       reinterpret_cast<double*>(blk + so.ring), S, bw, x, lane);
  double* need = p.need_scratch + (size_t)n * S;
#pragma unroll 1
  for (int e = lane; e < S; e += 32) need[e] = x[e];
  flags = __reduce_or_sync(kFull, flags);
  if (lane == 0 && flags && p.trace.flags) p.trace.flags[n] |= flags;
}

// ---------------------------------------------------------------------------
// pma_sr_band_kernel: the full SR = inv(I - gamma T) of a banded T, once at the end of a banded call, from the band
// factors pma_band_factor_kernel leaves in band_scratch.  One CTA per agent, thread c solves COLUMN c of the
// inverse (L y = e_c forward, U x = y backward): at step i every thread touches SR[i][c], so the S x S result is
// written (and the intermediate y read back) with fully coalesced rows and nothing but the factors has to be
// staged -- 21 KB of shared memory per CTA instead of the 101 KB of a row-per-thread solve that kept its S x S
// block on chip (2 CTAs per SM, 0.30 instructions / cycle / scheduler, profiles/r1_pma_v3_banded.txt).
// 2 S^2 bw operations instead of the S^3 of the dense Gauss-Jordan.
// ---------------------------------------------------------------------------
template <int BW>      // BW >= sr_band: length of the per-thread register window
__global__ void __launch_bounds__(512) pma_sr_band_kernel(const __grid_constant__ CobelPMAParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, bw = p.sr_band, W = 2 * bw + 1, tid = threadIdx.x;
  const int64_t n = blockIdx.x;
  constexpr int WP = 2 * BW + 2;                                   // padded factor row: entry [BW + d] = factor[j][j + d]
  double* fac = reinterpret_cast<double*>(smem);                   // [S][WP], zero-padded to the window length
  {
    const double* fg = p.band_scratch + (size_t)n * S * W;
    for (int e = tid; e < S * WP; e += blockDim.x) {
      const int j = e / WP, d = e - j * WP - BW;                   // d = column offset -BW .. BW + 1
      fac[e] = (d >= -bw && d <= bw) ? fg[(size_t)j * W + bw + d] : 0.0;
    }
  }
  __syncthreads();
  const int c = tid, i0 = tid & ~31;                               // a warp walks i from its first column on (y_i = 0 above)
  if (i0 >= S) return;
  double* col = p.SR + (size_t)n * S * S + min(c, S - 1);          // element i of this thread's column: col[i * S]
  const bool live = c < S;
  // The last BW solution entries live in a register window whose rotation is static: the loops advance in chunks
  // of BW fully unrolled steps, step u of a chunk writes slot u and reads y_{i-d} / x_{i+d} from slot (u - d) mod BW
  // (no shifting moves; the factors of a step are BW / 2 LDS.128).
  double w[BW];
#pragma unroll
  for (int d = 0; d < BW; ++d) w[d] = 0.0;
#pragma unroll 1
  for (int ib = i0; ib < S; ib += BW) {                            // L y = e_c (unit diagonal; multipliers l[i][i-d] at offset -d)
#pragma unroll
    for (int u = 0; u < BW; ++u) {
      const int i = ib + u;
      if (i < S) {
        const double* f = fac + (size_t)i * WP + BW;
        double acc = i == c ? 1.0 : 0.0;
#pragma unroll
        for (int d = 1; d <= BW; ++d) acc = fma(-f[-d], w[(u - d + 2 * BW) % BW], acc);
        if (live) col[(size_t)i * S] = acc;
        w[u] = acc;
      }
    }
  }
#pragma unroll
  for (int d = 0; d < BW; ++d) w[d] = 0.0;
  // y_i = 0 above the warp's first column; the loads of y run two steps ahead of the recurrence
  auto yld = [&](int i) -> double { return (live && i >= i0) ? col[(size_t)i * S] : 0.0; };
  double y0 = yld(S - 1), y1 = yld(S - 2);
#pragma unroll 1
  for (int ib = S - 1; ib >= 0; ib -= BW) {                        // U x = y (the diagonal holds 1 / pivot)
#pragma unroll
    for (int u = 0; u < BW; ++u) {
      const int i = ib - u;
      if (i >= 0) {
        const double* f = fac + (size_t)i * WP + BW;
        double acc = y0;
        y0 = y1;
        y1 = yld(i - 2);
#pragma unroll
        for (int d = 1; d <= BW; ++d) acc = fma(-f[d], w[(u - d + 2 * BW) % BW], acc);
        const double xi = acc * f[0];
        if (live) col[(size_t)i * S] = xi;
        w[u] = xi;
      }
    }
  }
}

// The caller's band guarantee on the initial T (a streaming read of T, once per banded call).
__global__ void __launch_bounds__(256) pma_band_check_kernel(const __grid_constant__ CobelPMAParams p) {
  const int S = p.world.n_states, bw = p.sr_band;
  const int64_t n = blockIdx.x;
  const double* Tg = p.T + (size_t)n * S * S;
  int bad = 0;
#pragma unroll 8
  for (int e = threadIdx.x; e < S * S; e += 256) {
    const int i = e / S, j = e - i * S;
    bad |= (abs(i - j) > bw && Tg[e] != 0.0) ? 1 : 0;
  }
  bad = __syncthreads_or(bad);
  if (threadIdx.x == 0 && bad && p.trace.flags) p.trace.flags[n] |= COBEL_FLAG_BAND_VIOLATION;
}

// ---------------------------------------------------------------------------
// Tie-pattern policy tables (CobelPMAParams.tab_*): for the two epsilon-greedy kinds get_action_probs depends only
// on idx = valid-action mask << A | tie pattern, so per distinct (kind, parameter) three tables of (1 << 2A) rows
// of A doubles are built once per call -- with exactly the operations of probs_row / select_action_warp:
//   raw   get_action_probs(v, mask)                                  policy/greedy.py:60-88, 117-147
//   norm  raw / np.sum(raw)       (action_probs_batch)               memory/pma.py:423-450
//   cdf   cumsum(raw) / cumsum(raw)[-1], last entry 2.0 (never <= u) policy/greedy.py:58
// ---------------------------------------------------------------------------
template <int A>
struct PolTab {
  static constexpr int kIdx = 1 << (2 * A);
  static constexpr int kDoubles = 3 * kIdx * A;
  const double* base;
  COBEL_DEV const double* raw(int idx) const { return base + idx * A; }
  COBEL_DEV const double* norm(int idx) const { return base + (kIdx + idx) * A; }
  COBEL_DEV const double* cdf(int idx) const { return base + (2 * kIdx + idx) * A; }
};

template <int A>
__global__ void __launch_bounds__(256) pma_policy_table_kernel(const int32_t* __restrict__ kind, const double* __restrict__ param,
                                                               double* out) {
  constexpr int kIdx = PolTab<A>::kIdx;
  const int c = blockIdx.x;
  if (c == (int)gridDim.x - 1) {
    // last block: Generator.choice(p = ones(k) / k) for k = 1..32 (memory/pma.py:252-254), row k-1 holds the bin
    // edges cdf_m / cdf_k, m < k-1 (cdf_m = m+1 sequential additions of fl(1/k)); other entries 2.0 (never <= u)
    double* tie = out + (size_t)c * PolTab<A>::kDoubles;
    if (threadIdx.x < 32) {
      const int k = threadIdx.x + 1;
      const double pk = xdiv(1.0, (double)k);
      double ck = 0.0;
      for (int m = 0; m < k; ++m) ck = xadd(ck, pk);
      double cm = 0.0;
      for (int m = 0; m < 32; ++m) {
        cm = xadd(cm, pk);
        tie[threadIdx.x * 32 + m] = m < k - 1 ? xdiv(cm, ck) : 2.0;
      }
    }
    return;
  }
  const int kd = kind[c];
  const double par = param[c];
  double* raw = out + (size_t)c * PolTab<A>::kDoubles;
  double* norm = raw + kIdx * A;
  double* cdf = norm + kIdx * A;
  for (int idx = threadIdx.x; idx < kIdx; idx += blockDim.x) {
    const uint32_t mask = (uint32_t)idx >> A, ties = (uint32_t)idx & ((1u << A) - 1u);
    const bool ok = ties != 0 && (ties & ~mask) == 0 && kd != COBEL_POLICY_SOFTMAX;
    double p[A], pn[A], cd[A];
#pragma unroll
    for (int a = 0; a < A; ++a) { p[a] = 0.0; pn[a] = 0.0; cd[a] = 2.0; }
    if (ok) {
      const int nv = __popc(mask), k = __popc(ties);
      const double tie = xdiv(xsub(1.0, par), (double)k);
      double top, low;
      if (kd == COBEL_POLICY_EPS_GREEDY) {
        const double base = xdiv(par, (double)nv);
        top = xadd(base, tie); low = xadd(base, 0.0);
      } else {
        const int d = nv - k > 1 ? nv - k : 1;
        top = xadd(tie, 0.0); low = xadd(0.0, xdiv(par, (double)d));
      }
#pragma unroll
      for (int a = 0; a < A; ++a) p[a] = (mask >> a & 1u) ? ((ties >> a & 1u) ? top : low) : 0.0;
      double s = p[0], c2 = p[0];
      cd[0] = c2;
#pragma unroll
      for (int a = 1; a < A; ++a) { s = xadd(s, p[a]); c2 = xadd(c2, p[a]); cd[a] = c2; }
#pragma unroll
      for (int a = 0; a < A; ++a) pn[a] = xdiv(p[a], s);
      if (c2 != 1.0) {
#pragma unroll
        for (int a = 0; a < A; ++a) cd[a] = xdiv(cd[a], c2);
      }
      cd[A - 1] = 2.0;
    }
#pragma unroll
    for (int a = 0; a < A; ++a) { raw[idx * A + a] = p[a]; norm[idx * A + a] = pn[a]; cdf[idx * A + a] = cd[a]; }
  }
}

// read-only row of A doubles from a 16-byte aligned global table (A even -> LDG.128)
template <int A>
COBEL_DEV void ldg_row(const double* r, double (&v)[A]) {
  if constexpr (A % 2 == 0) {
#pragma unroll
    for (int x = 0; x < A; x += 2) {
      const double2 t = __ldg(reinterpret_cast<const double2*>(r + x));
      v[x] = t.x; v[x + 1] = t.y;
    }
  } else {
#pragma unroll
    for (int x = 0; x < A; ++x) v[x] = __ldg(r + x);
  }
}

// table row of a Q row: valid mask << A | (valid entries equal to the maximum over the valid entries)
template <int A>
COBEL_DEV int tie_index(const double (&v)[A], uint32_t mb) {
  const double ninf = -__longlong_as_double(0x7FF0000000000000ll);
  double w[A];
#pragma unroll
  for (int a = 0; a < A; ++a) w[a] = (mb >> a & 1u) ? v[a] : ninf;
  const double m = row_max<A>(w);
  uint32_t ties = 0;
#pragma unroll
  for (int a = 0; a < A; ++a) ties |= (w[a] == m ? 1u : 0u) << a;
  return (int)((mb << A) | ties);
}

// Policy.select_action from the cdf table: the number of bin edges <= u (every lane computes the same)
template <int A>
COBEL_DEV int select_action_tab(const double (&v)[A], uint32_t mb, const PolTab<A>& tab, double u) {
  double c[A];
  ldg_row<A>(tab.cdf(tie_index<A>(v, mb)), c);
  int a = 0;
#pragma unroll
  for (int x = 0; x < A - 1; ++x) a += c[x] <= u ? 1 : 0;
  return a;
}

// ---------------------------------------------------------------------------
// Utilities are kept as order-preserving integer keys: (hi signed, lo unsigned) compares like the double, equal
// keys <=> equal doubles (-0.0 is canonicalised to +0.0 first; utilities are never NaN).  A warp maximum is then
// two REDUX instructions instead of a five-level fp64 shuffle butterfly.
// ---------------------------------------------------------------------------
COBEL_DEV int2 key_of(double v) {                     // .x = lo, .y = hi
  v = xadd(v, 0.0);
  int hi = __double2hiint(v), lo = __double2loint(v);
  const int s = hi >> 31;
  return make_int2(lo ^ s, hi ^ (s & 0x7FFFFFFF));
}
COBEL_DEV double key_value(int2 k) {
  const int s = k.y >> 31;
  return __hiloint2double(k.y ^ (s & 0x7FFFFFFF), k.x ^ s);
}
constexpr int kKeyMinHi = (int)0x80000000;            // below the key of every double (-inf included)
COBEL_DEV int2 warp_max_key(int2 k) {
  const int mh = __reduce_max_sync(kFull, k.y);
  const unsigned ml = __reduce_max_sync(kFull, k.y == mh ? (unsigned)k.x : 0u);
  return make_int2((int)ml, mh);
}

// ---------------------------------------------------------------------------
// pma_main_kernel: one warp per agent.
// ---------------------------------------------------------------------------
struct MainSmem {      // byte offsets inside one agent's shared-memory block
  int q, mr, need, pk, mbits, ukey, poff, pitems, list, perf, dst, rs, bar, bytes;
  int np;              // utility entries padded to a multiple of 32 (chunks of one entry per lane)
  static constexpr int kListCap = 256;     // stale-gain list; larger sets fall back to a full pass
  __host__ __device__ MainSmem(int S, int A) {
    const int N = S * A;
    np = (N + 31) & ~31;
    q = 0;
    mr = q + N * 8;
    need = mr + N * 8;
    pk = need + ((S + 1) & ~1) * 8;
    mbits = pk + N * 2;
    // from here on: buffers that are dead between replay calls
    ukey = (mbits + S + 7) & ~7;
    poff = ukey + np * 8;
    pitems = poff + ((S + 3) & ~1) * 4;
    list = pitems + N * 2;
    perf = list + kListCap * 2;
    dst = perf + (kMaxSeq + 2) * 2;
    rs = (dst + (kMaxSeq + 2) * 2 + 7) & ~7;
    bar = rs + (kMaxSeq + 2) * 8;            // mbarrier of the bulk stage-in
    bytes = (bar + 8 + 15) & ~15;
  }
};

// launch phases of pma_main_kernel: [end-of-trial replay of the previous trial] [reset] [n_trials x (start-of-trial
// replay + online steps)].  With replays on, update_sr sits between a trial's steps and its end replay, so a launch
// runs one trial at most and the per-agent state travels in `carry`.
struct MainPhase {
  int init_carry;       // first launch of a run: reset the per-agent carry
  int end_replay;       // replay(last) of the previous trial first
  int reset;            // draw the start state of the next trial (else it comes from carry[4])
  int n_trials;         // trials run by this launch (several only without replays; later ones reset themselves)
  int trial_first;      // index of the first trial run by this launch
  int scratch_need;     // banded update_sr: both replays read their need vector from need_scratch (1: its first plane;
                        // 2: the end replay from the first, the start replay from the second plane)
};

// PLAIN = epsilon-greedy agent and memory policies from the tie-pattern tables, training with replay,
// deterministic world, no optional trace buffers, generated stream: the per-row policy evaluation (fp64
// divisions, exp) and the per-step checks are compiled out.
// BIG = more than 1024 one-step backups or more than 160 states (up to 2048 / 512: 20x20 with 4 actions): two chunk
// maxima per lane and a longer register window for the T row of a step; the common sizes keep the lean code.
template <int A, bool PLAIN, bool BIG = false>
__global__ void __launch_bounds__(kMainWarps * 32, BIG ? 1 : 4) pma_main_kernel(const __grid_constant__ CobelPMAParams p,
                                                                      const __grid_constant__ MainPhase ph) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, K = p.world.n_starts, N = S * A, B = p.batch;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n = (int64_t)blockIdx.x * kMainWarps + warp;
  if (n >= p.n_agents) return;                         // whole warp leaves; no block-wide barrier is used
  const MainSmem so(S, A);
  unsigned char* blk = smem + (size_t)warp * so.bytes;
  double* Q = reinterpret_cast<double*>(blk + so.q);         // [s][a]
  double* Mr = reinterpret_cast<double*>(blk + so.mr);       // [s][a]
  int2* ukey = reinterpret_cast<int2*>(blk + so.ukey);       // [a*S+s] key of gain * need * update_mask of the one-step backups
  double* need = reinterpret_cast<double*>(blk + so.need);   // [s] need of the current replay call
  int32_t* poff = reinterpret_cast<int32_t*>(blk + so.poff); // [S+2] CSR: backups that bootstrap from row t are pitems[poff[t+1] .. poff[t+2])
  uint16_t* Pk = reinterpret_cast<uint16_t*>(blk + so.pk);   // [s][a] M.states | update_mask << 13 | M.terminals << 15
  uint16_t* pitems = reinterpret_cast<uint16_t*>(blk + so.pitems); // CSR items (flat indices a*S+s)
  uint16_t* list = reinterpret_cast<uint16_t*>(blk + so.list);     // flat indices of the stale gains
  uint16_t* perf = reinterpret_cast<uint16_t*>(blk + so.perf); // performed updates of this replay call
  uint16_t* dst = reinterpret_cast<uint16_t*>(blk + so.dst);   // states whose Q row changed in the last update
  double* rs = reinterpret_cast<double*>(blk + so.rs);         // M.rewards of the candidate sequence's elements
  uint8_t* mbits = blk + so.mbits;                             // [s] valid-action bits (all ones if unmasked)
  constexpr int kSt = 0x1FFF, kUm = 0x2000;
  static_assert(!(PLAIN && BIG), "the large-state instantiation is the generic kernel");
  constexpr int kH = BIG ? 2 : 1;                              // chunk maxima per lane: chunk c lives in lane c & 31, slot c >> 5
  constexpr int kTrow = BIG ? 16 : 5;                          // T-row entries per lane (S <= 512 / 160)
  const int nch = so.np >> 5;                                  // chunks of 32 consecutive utilities (at most 32 kH)
  // flat backup index i = a*S + s (the reference's order, memory/pma.py:205) -> a, s, s*A + a without integer
  // division: i < 2048 and S <= 512, so (i * ceil(2^24 / S)) >> 24 == i / S exactly (and i * ceil(.) < 2^28)
  const uint32_t magicS = ((1u << 24) + (uint32_t)S - 1u) / (uint32_t)S;
  auto act_of = [&](int i) -> int { return (int)(((uint32_t)i * magicS) >> 24); };
  auto st_of = [&](int i) -> int { return i - act_of(i) * S; };
  auto sa_of = [&](int i) -> int { const int a_ = act_of(i); return (i - a_ * S) * A + a_; };

  const size_t g0 = (size_t)n * N;
  double* Tg = p.T + (size_t)n * S * S;
  const double* SRg = p.SR + (size_t)n * S * S;
  const uint8_t* amask = p.action_mask ? p.action_mask + n * p.mask_agent_stride : nullptr;
  // Stage-in: Q and M.rewards arrive by two bulk asynchronous copies (TMA 1-D path) issued by lane 0, while the lanes
  // pack M.states | update_mask | M.terminals; rows that are not 16-byte multiples take the plain loop.
  uint64_t* bar = reinterpret_cast<uint64_t*>(blk + so.bar);
  const bool bulk = (N & 1) == 0 && aligned16(p.Q) && aligned16(p.Mr);
  if (bulk) {
    if (lane == 0) {
      mbar_init(bar, 1);
      mbar_fence_init();
      mbar_expect_tx(bar, 2u * (unsigned)N * 8u);
      bulk_load(Q, p.Q + g0, (unsigned)N * 8u, bar);
      bulk_load(Mr, p.Mr + g0, (unsigned)N * 8u, bar);
    }
  } else {
#pragma unroll 1
    for (int e = lane; e < N; e += 32) { Q[e] = p.Q[g0 + e]; Mr[e] = p.Mr[g0 + e]; }
  }
#pragma unroll 4
  for (int e = lane; e < N; e += 32) {
    const int s_ = e / A, a_ = e - s_ * A;
    Pk[e] = (uint16_t)(p.Ms[g0 + e] | (p.update_mask[g0 + a_ * S + s_] ? kUm : 0) | ((p.Mt[g0 + e] ? 1 : 0) << 15));
  }
#pragma unroll 1
  for (int e = lane; e < S; e += 32) {
    uint32_t mb = (1u << A) - 1u;
    if (amask) {
      mb = 0;
      for (int a = 0; a < A; ++a) mb |= (amask[e * A + a] ? 1u : 0u) << a;
    }
    mbits[e] = (uint8_t)mb;
  }
  const double* powsr = p.pow_gamma_sr + n * p.pow_stride;     // float(M.gamma) ** k
  const double* powq = p.pow_gamma_q + n * p.pow_stride;       // float(M.gamma_q) ** k
  constexpr int kPol = PLAIN ? COBEL_POLICY_EPS_GREEDY : -1;
  const int mkind = p.mem_policy.kind;
  const double mpar = p.mem_policy.param[n];
  // tie-pattern tables of the agent's and the memory's policy (PLAIN: both guaranteed by the host)
  const bool have_tab = PLAIN || (p.n_tab > 0 && A <= 4);
  PolTab<A> tabA{nullptr}, tabM{nullptr};
  if (have_tab) {
    const int ta = p.tab_of_agent ? p.tab_of_agent[2 * n] : 0;
    const int tm = p.tab_of_agent ? p.tab_of_agent[2 * n + 1] : p.n_tab - 1;
    tabA.base = p.tab_scratch + (size_t)ta * PolTab<A>::kDoubles;
    tabM.base = p.tab_scratch + (size_t)tm * PolTab<A>::kDoubles;
  }
  const double* tie_cdf = have_tab ? p.tab_scratch + (size_t)p.n_tab * PolTab<A>::kDoubles : nullptr;   // [32][32]
  const bool useA = PLAIN || (have_tab && p.policy.kind != COBEL_POLICY_SOFTMAX);
  const bool useM = PLAIN || (have_tab && mkind != COBEL_POLICY_SOFTMAX);
  // per-row evaluation (generic kernel only): cached quotients par/n and (1-par)/n of the memory policy
  double qpar[A], qom[A];
  if (!PLAIN) {
#pragma unroll
    for (int a = 0; a < A; ++a) { qpar[a] = xdiv(mpar, (double)(a + 1)); qom[a] = xdiv(xsub(1.0, mpar), (double)(a + 1)); }
  }
  __syncwarp();

  int64_t* carry = p.carry + n * 8;           // [0] last state (-1: timed out)  [1] steps  [2] replayed  [3] replay calls  [4] start state
  int64_t c_last = ph.init_carry ? -1 : carry[0];
  int64_t nsteps = ph.init_carry ? 0 : carry[1], nrep = ph.init_carry ? 0 : carry[2], ncalls = ph.init_carry ? 0 : carry[3];
  const int64_t nsteps0 = nsteps, nrep0 = nrep;

  DrawWindowT<!PLAIN, true> win; win.init(p.stream, n, (uint64_t)p.stream.draw_count[n]);
  const double lr = p.lr[n], gamma = p.gamma[n], mlr = p.mem_lr[n];
  const double lrq = p.lr_q[n], gq = p.gamma_q[n];
  const double min_gain = p.min_gain;
  const bool original = p.min_gain_original != 0;
  const int opt = PLAIN ? 0 : p.options;        // COBEL_PMA_OPT_* (the PLAIN kernel is built for none of them)
  PolicyTab pt, mpt;
  if (!PLAIN) { pt.init(p.policy.kind, p.policy.param[n], lane); mpt.init(mkind, mpar, lane); }
  const bool learn = PLAIN || p.learn != 0;
  const bool do_replay = PLAIN || (learn && !p.no_replay);
  const CobelTrace& tr = p.trace;
  int flags = 0;
  // certificate: the smallest relative gap (umax - u2) / |umax| between the two largest distinct utilities, kept
  // as a fraction (one division per launch instead of one per selection)
  double gap_num = __longlong_as_double(0x7FF0000000000000ll), gap_den = 1.0;

  // utility of a backup with gain g at (s, a): gain * need * update_mask (memory/pma.py:247-249), as a key
  auto util_key = [&](double g, int s, int a) -> int2 {
    const double gn = xmul(g, need[s]);
    if (opt & COBEL_PMA_OPT_KEEP_BARRIERS) return key_of(gn);       // ignore_barriers False, memory/pma.py:248-249
    return key_of(xmul(gn, (Pk[s * A + a] & kUm) ? 1.0 : 0.0));
  };

  // PMAMemory.replay, memory/pma.py:168-267.  nsrc = the need vector in HBM (an SR row or the stationary
  // need); nullptr: need[] has been filled in place by the banded solver.
  auto replay = [&](const double* nsrc) {
    if (nsrc) {
#pragma unroll 1
      for (int e = lane; e < S; e += 32) need[e] = nsrc[e];
    }
    if (opt & COBEL_PMA_OPT_EQUAL_NEED) {                              // need.fill(1), memory/pma.py:244-245
      __syncwarp();
#pragma unroll 1
      for (int e = lane; e < S; e += 32) need[e] = 1.0;
    }
    // CSR of the backups grouped by the Q row they bootstrap from (M.states does not change during a replay).
    // Only backups with M.terminals != 0 take part: a zero flag multiplies the bootstrap value away
    // (memory/pma.py:362-363), so their gain does not depend on that row -- in particular the never-experienced
    // backups, which all point at state 0.  The backups that read Q row t are row t itself and group t.
#pragma unroll 1
    for (int e = lane; e < S + 2; e += 32) poff[e] = 0;
    if (lane < so.np - N) ukey[N + lane] = make_int2(0, kKeyMinHi);   // padding of the last chunk never wins
    __syncwarp();
#pragma unroll 1
    for (int e = lane; e < N; e += 32) { const uint16_t pk = Pk[e]; if (pk >> 15) atomicAdd(&poff[(pk & kSt) + 1], 1); }
    __syncwarp();
    {                                               // inclusive prefix sum of poff[1..S]: a segment per lane + a warp scan
      const int seg = (S + 31) >> 5, b0 = lane * seg;
      int sum = 0;
#pragma unroll 1
      for (int x = 0; x < seg; ++x) { const int t = b0 + x; if (t < S) sum += poff[t + 1]; }
      int incl = sum;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(kFull, incl, d); if (lane >= d) incl += o; }
      int run = incl - sum;
#pragma unroll 1
      for (int x = 0; x < seg; ++x) { const int t = b0 + x; if (t < S) { run += poff[t + 1]; poff[t + 1] = run; } }
      const int tot = __shfl_sync(kFull, incl, 31);
      if (lane == 0) poff[S + 1] = tot;
    }
    __syncwarp();
#pragma unroll 1
    for (int e = lane; e < N; e += 32) {            // fill each group from its back: poff[t+1] ends as the start of group t
      const uint16_t pk = Pk[e];
      if (pk >> 15) {
        const int s_ = e / A, a_ = e - s_ * A;
        pitems[atomicSub(&poff[(pk & kSt) + 1], 1) - 1] = (uint16_t)(a_ * S + s_);
      }
    }
    __syncwarp();
    int count = 0, last_seq = 0, ndst = -1;          // ndst < 0: first iteration, every backup is stale
    unsigned dirty[kH];                              // chunks whose maximum has to be recomputed
    int cm_hi[kH]; unsigned cm_lo[kH];               // lane l, slot h: the largest key of chunk 32 h + l
#pragma unroll
    for (int h = 0; h < kH; ++h) {
      const int left = nch - 32 * h;
      dirty[h] = left >= 32 ? kFull : (left > 0 ? (1u << left) - 1u : 0u);
      cm_hi[h] = kKeyMinHi; cm_lo[h] = 0;
    }
    unsigned seqmask = 0;                            // lane w: bits of the states 32 w .. 32 w + 31 in performed[last_seq:]
    for (int it = 0; it < B; ++it) {
      // ---- (1) extension of the current sequence (memory/pma.py:219-235) -------------------------
      // The candidate sequence is performed[last_seq:] + [ext]: it is read in place from perf[] (perf[count] holds
      // the candidate until the chosen update overwrites it); seqmask = the states of performed[last_seq:].
      int ext = -1, clen = 0, seq_base = 0;
      if (count > 0) {
        const int lp = perf[count - 1];
        ext = Pk[sa_of(lp)] & kSt;                          // next_state of the last update
        const bool loop = (__shfl_sync(kFull, seqmask, ext >> 5) >> (ext & 31)) & 1u;
        if (!loop || (opt & COBEL_PMA_OPT_ALLOW_LOOPS)) {
          win.ensure(2, lane);
          double row[A];
          load_row<A>(Q + ext * A, row);
          const double u = win.next();
          const int ea = (PLAIN || useM) ? select_action_tab<A>(row, mbits[ext], tabM, u)
                                         : select_action_warp<A, kPol>(row, mbits[ext], mpt, u, lane);
          ext += ea * S;
          clen = count - last_seq + 1;
          seq_base = last_seq;
        } else {
          seq_base = count;                                 // failed extension: one-step(ext, action 0)
        }
        if (lane == 0) perf[count] = (uint16_t)ext;
        __syncwarp();                                       // seq[] is read by all lanes in (2)
      }
      const uint16_t* seq = perf + seq_base;
      // ---- (2) work list of this iteration: the one-step backups whose gain is stale (they read a Q row changed
      // by the previous update; everything on the first iteration) followed by the elements of the candidate
      // n-step sequence.  Both kinds are "the gain of moving Q[s,a] towards a target" (memory/pma.py:269-386):
      //   one-step   target = M.rewards + gamma_q max Q[s'] M.terminals, probabilities p / sum(p), clipped
      //   n-step     target = discounted reward sum + bootstrap, raw probabilities, clipped per element if 'original'
      // so ONE evaluation pass serves both (lane = work item).
      int nd = 0;
      bool full = ndst < 0;
#pragma unroll 1
      for (int d = 0; d < ndst && !full; ++d) {
        const int t = dst[d];
        const int p0 = poff[t + 1], np = poff[t + 2] - p0;
        if (nd + A + np <= MainSmem::kListCap) {
#pragma unroll 1
          for (int x = lane; x < A + np; x += 32) list[nd + x] = x < A ? (uint16_t)(x * S + t) : pitems[p0 + x - A];
          nd += A + np;
        } else {
          full = true;
        }
      }
      const int n1 = full ? N : nd;
      const int nseq = ext >= 0 ? (clen > 0 ? clen : 1) : 0;
      double fv = 0.0;
      if (nseq) {
#pragma unroll 1
        for (int j = lane; j < nseq; j += 32) rs[j] = Mr[sa_of(seq[j])];
        const uint16_t lpk = Pk[sa_of(seq[nseq - 1])];
        double lrow[A];
        load_row<A>(Q + (lpk & kSt) * A, lrow);
        fv = xmul(row_max<A>(lrow), (lpk >> 15) ? 1.0 : 0.0);
      }
      __syncwarp();
      double total = 0.0;                                  // gain of the candidate: its elements' gains added in order
      unsigned myd[kH];
#pragma unroll
      for (int h = 0; h < kH; ++h) myd[h] = 0;
#pragma unroll 1
      for (int j0 = 0; j0 < n1 + nseq; j0 += 32) {
        const int j = j0 + lane;
        const bool one = j < n1;
        double g = 0.0;
        if (j < n1 + nseq) {
          const int e = j - n1;
          const int i = one ? (full ? j : list[j]) : seq[e];
          const int a = act_of(i), s = i - a * S;
          double q[A], qn[A], po[A], pn[A], t[A];
          load_row<A>(Q + s * A, q);
          double target;
          if (one) {
            const uint16_t pk = Pk[s * A + a];
            double tr_[A];
            load_row<A>(Q + (pk & kSt) * A, tr_);
            target = xadd(Mr[s * A + a], xmul(xmul(gq, row_max<A>(tr_)), (pk >> 15) ? 1.0 : 0.0));
          } else {
            double r = 0.0;
#pragma unroll 1
            for (int f = 0; f < nseq - e; ++f) r = xadd(r, xmul(rs[e + f], powsr[f]));
            target = xadd(r, xmul(fv, powq[nseq - e]));
          }
          {
            const double qa = pick<A>(q, a);
            const double upd = xadd(qa, xmul(lrq, xsub(target, qa)));
#pragma unroll
            for (int c = 0; c < A; ++c) qn[c] = c == a ? upd : q[c];
          }
          const uint32_t mb = mbits[s];
          if (PLAIN || useM) {
            const double* tb = one ? tabM.norm(0) : tabM.raw(0);
            ldg_row<A>(tb + tie_index<A>(q, mb) * A, po);
            ldg_row<A>(tb + tie_index<A>(qn, mb) * A, pn);
          } else {
            probs_row<A>(q, mb, mkind, mpar, qpar, qom, po);
            probs_row<A>(qn, mb, mkind, mpar, qpar, qom, pn);
            if (one) {
              const double so_ = sum_seq<A>(po), sn_ = sum_seq<A>(pn);
              // p / sum(p): x / 1.0 == x, so the (frequent) exactly-normalised case skips the divisions
              if (sn_ != 1.0) {
#pragma unroll
                for (int c = 0; c < A; ++c) pn[c] = pdiv(pn[c], sn_);
              }
              if (so_ != 1.0) {
#pragma unroll
                for (int c = 0; c < A; ++c) po[c] = pdiv(po[c], so_);
              }
            }
          }
#pragma unroll
          for (int c = 0; c < A; ++c) t[c] = xmul(pn[c], qn[c]);
          const double gnew = sum_seq<A>(t);
#pragma unroll
          for (int c = 0; c < A; ++c) t[c] = xmul(po[c], qn[c]);
          g = xsub(gnew, sum_seq<A>(t));
          if (one) {
            g = g > min_gain ? g : min_gain;
            if (opt & COBEL_PMA_OPT_EQUAL_GAIN) g = 1.0;               // gain.fill(1), memory/pma.py:241-242
            ukey[i] = util_key(g, s, a);
            if (!BIG || (i >> 10) == 0) myd[0] |= 1u << ((i >> 5) & 31);
            else myd[kH - 1] |= 1u << ((i >> 5) & 31);
          } else if (original) {
            g = g > min_gain ? g : min_gain;
          }
        }
        if (nseq) {                                        // gain += step_gain, in sequence order
          const int lo = n1 - j0 > 0 ? n1 - j0 : 0, hi = n1 + nseq - j0 < 32 ? n1 + nseq - j0 : 32;
#pragma unroll 1
          for (int l = lo; l < hi; ++l) total = xadd(total, shfl_f64(g, l));
        }
      }
#pragma unroll
      for (int h = 0; h < kH; ++h) dirty[h] |= __reduce_or_sync(kFull, myd[h]);
      __syncwarp();
      double gext = total > min_gain ? total : min_gain;
      if (opt & COBEL_PMA_OPT_EQUAL_GAIN) gext = 1.0;
      // ---- (4) arg-max of the utilities with exact ties (memory/pma.py:247-254); the candidate's
      // n-step gain overrides the one-step entry `ext` for this iteration only
      int2 saved = make_int2(0, 0);
      if (ext >= 0) {
        const int ea = act_of(ext), es = ext - ea * S;
        saved = ukey[ext];
        __syncwarp();
        if (lane == 0) ukey[ext] = util_key(gext, es, ea);
        dirty[BIG ? (ext >> 10) : 0] |= 1u << ((ext >> 5) & 31);
        __syncwarp();
      }
      // chunk maxima are kept across iterations: only the chunks that received a new utility are reduced again
#pragma unroll
      for (int h = 0; h < kH; ++h) {
        while (dirty[h]) {
          const int c = __ffs(dirty[h]) - 1;
          dirty[h] &= dirty[h] - 1;
          const int2 m = warp_max_key(ukey[(h * 32 + c) * 32 + lane]);
          if (lane == c) { cm_hi[h] = m.y; cm_lo[h] = (unsigned)m.x; }
        }
      }
      int2 cmine[kH];
#pragma unroll
      for (int h = 0; h < kH; ++h) cmine[h] = make_int2((int)cm_lo[h], h * 32 + lane < nch ? cm_hi[h] : kKeyMinHi);
      int2 lbest = cmine[0];
      if (kH > 1 && (cmine[kH - 1].y > lbest.y || (cmine[kH - 1].y == lbest.y && (unsigned)cmine[kH - 1].x > (unsigned)lbest.x)))
        lbest = cmine[kH - 1];
      const int2 umax = warp_max_key(lbest);
      // the largest utility below the maximum: over the other chunks' maxima and the rest of the winning chunks
      bool cwin[kH];
      unsigned tch[kH];
      int2 lsec = make_int2(0, kKeyMinHi);
#pragma unroll
      for (int h = 0; h < kH; ++h) {
        cwin[h] = cmine[h].y == umax.y && cmine[h].x == umax.x;          // chunk holds a maximum
        tch[h] = __ballot_sync(kFull, cwin[h]);
        if (!cwin[h] && (cmine[h].y > lsec.y || (cmine[h].y == lsec.y && (unsigned)cmine[h].x > (unsigned)lsec.x))) lsec = cmine[h];
      }
      int2 second = warp_max_key(lsec);
      // ties in flat-index order: lane l, slot h keeps the tie ballot of chunk 32 h + l
      unsigned mytb[kH];
      unsigned onlyb = 0;
      const int c0 = (tch[0] || kH == 1) ? __ffs(tch[0]) - 1 : 32 + __ffs(tch[kH - 1]) - 1;
#pragma unroll
      for (int h = 0; h < kH; ++h) {
        mytb[h] = 0;
        unsigned t = tch[h];
        while (t) {
          const int c = __ffs(t) - 1;
          t &= t - 1;
          const int2 k = ukey[(h * 32 + c) * 32 + lane];
          const bool eq = k.y == umax.y && k.x == umax.x;
          const unsigned b = __ballot_sync(kFull, eq);
          const int2 r2 = warp_max_key(eq ? make_int2(0, kKeyMinHi) : k);
          if (r2.y > second.y || (r2.y == second.y && (unsigned)r2.x > (unsigned)second.x)) second = r2;
          mytb[h] = lane == c ? b : mytb[h];
          if (!onlyb) onlyb = b;
        }
      }
      int mycnt = 0;
#pragma unroll
      for (int h = 0; h < kH; ++h) mycnt += __popc(mytb[h]);
      const int ktot = __reduce_add_sync(kFull, mycnt);
      {
        const double vmax = key_value(umax);
        if (second.y != kKeyMinHi && vmax != 0.0) {
          const double v2 = key_value(second);
          if (v2 > -1e300) {
            const double num = xsub(vmax, v2), den = fabs(vmax);
            if (num * gap_den < gap_num * den) { gap_num = num; gap_den = den; }
          }
        }
      }
      win.ensure(1, lane);
      const double u = win.next();
      int chosen;
      if (ktot == 1) {
        chosen = c0 * 32 + __ffs(onlyb) - 1;
      } else {
        // Generator.choice(p = ties / k): cdf_m = m-fold sequential sum of fl(1/k), normalised by cdf_k; the pick is
        // the number of bin edges <= u (tabulated per k <= 32 next to the policy tables)
        int pick;
        if ((PLAIN || have_tab) && ktot <= 32) {
          const double edge = __ldg(tie_cdf + (ktot - 1) * 32 + lane);
          pick = __popc(__ballot_sync(kFull, edge <= u));
        } else {
          pick = ktot - 1;
          const double pk_ = pdiv(1.0, int_to_f64(ktot));
          double ck = 0.0;
#pragma unroll 1
          for (int m = 0; m < ktot; ++m) ck = xadd(ck, pk_);
          double c = 0.0;
#pragma unroll 1
          for (int m = 0; m < ktot; ++m) {
            c = xadd(c, pk_);
            if (pdiv(c, ck) > u) { pick = m; break; }
          }
        }
        // the pick-th tie in flat-index order: walk the winning chunks (ascending) until their tie counts cover it
        chosen = 0;
        int base = 0;
        bool found = false;
#pragma unroll
        for (int h = 0; h < kH; ++h) {
          unsigned tc = tch[h];
          while (tc && !found) {
            const int c = __ffs(tc) - 1;
            tc &= tc - 1;
            const unsigned b = __shfl_sync(kFull, mytb[h], c);
            const int nb = __popc(b);
            if (pick < base + nb) {
              const unsigned sel = __ballot_sync(kFull, (b >> lane & 1u) && __popc(b & ((1u << lane) - 1u)) == pick - base);
              chosen = (h * 32 + c) * 32 + __ffs(sel) - 1;
              found = true;
            }
            base += nb;
          }
        }
      }
      if (ext >= 0) {
        __syncwarp();
        if (lane == 0) ukey[ext] = saved;
        dirty[BIG ? (ext >> 10) : 0] = 1u << ((ext >> 5) & 31);
      }
      // ---- (5) apply the chosen (n-step) update: PMAMemory.update_q, memory/pma.py:452-496 --------
      {
        const bool use_seq = clen > 0 && chosen == ext;
        const int nseq5 = use_seq ? clen : 1;
        const uint16_t* sq = use_seq ? seq : perf + count;
        double fv5 = fv;                              // the candidate's bootstrap value is still valid (Q unchanged)
        if (!use_seq) {
          const int csa = sa_of(chosen);
          if (lane == 0) { perf[count] = (uint16_t)chosen; rs[0] = Mr[csa]; }
          const uint16_t lpk = Pk[csa];
          double lrow[A];
          load_row<A>(Q + (lpk & kSt) * A, lrow);
          fv5 = xmul(row_max<A>(lrow), (lpk >> 15) ? 1.0 : 0.0);
        }
        __syncwarp();
        bool ok = true;                               // n >= 2: every transition must be non-terminal & experienced
        if (nseq5 >= 2) {
          bool bad = false;
#pragma unroll 1
          for (int j = lane; j < nseq5; j += 32) { const int k = sq[j]; bad |= (Pk[sa_of(k)] >> 15) == 0; }
          ok = !__any_sync(kFull, bad);
        }
        ndst = 0;
        // replay_td of this update (slot nrep + count of replay_idx) is the td of the sequence's last element, the
        // experience that replay_idx names; NaN when the n-step update aborts (no element is updated then).  The
        // elements return their td instead of storing it, so the lambda captures nothing new: capturing the trace or
        // the counters by reference there made the compiler keep the BIG kernel's locals in a local-memory frame.
        double last_td = __longlong_as_double(0x7FF8000000000000ll);
        if (ok) {
          auto update_element = [&](int j) -> double {
            const int i = sq[j];
            const int a = act_of(i), s = i - a * S;
            double r = 0.0;
#pragma unroll 1
            for (int f = 0; f < nseq5 - j; ++f) r = xadd(r, xmul(rs[j + f], powq[f]));
            double td = xadd(r, xmul(fv5, powq[nseq5 - j]));
            const double q = Q[s * A + a];
            td = xsub(td, q);
            Q[s * A + a] = xadd(q, xmul(lrq, td));
            dst[j] = (uint16_t)s;
            return td;
          };
          if (opt & COBEL_PMA_OPT_ALLOW_LOOPS) {      // a sequence may revisit (s, a): in order, like the reference's loop
            if (lane == 0) {
#pragma unroll 1
              for (int j = 0; j < nseq5; ++j) last_td = update_element(j);
            }
          } else {                                    // the states of a sequence are distinct: one element per lane
#pragma unroll 1
            for (int j = lane; j < nseq5; j += 32) last_td = update_element(j);
          }
          ndst = nseq5;
        }
        if constexpr (!PLAIN) {
          // the lane that updated the last element (lane 0 for the in-order loop and for an aborted update)
          const int owner = (ok && !(opt & COBEL_PMA_OPT_ALLOW_LOOPS)) ? (nseq5 - 1) & 31 : 0;
          if (tr.replay_td && lane == owner) {
            if (nrep + count < tr.replay_cap) tr.replay_td[n * tr.replay_cap + nrep + count] = last_td;
            else flags |= COBEL_FLAG_TRACE_OVERFLOW;
          }
        }
        ++count;
        const int cs = st_of(chosen);
        if (ext != chosen) { last_seq = it; seqmask = 0; }
        if (lane == (cs >> 5)) seqmask |= 1u << (cs & 31);
        __syncwarp();
      }
    }
    if (!PLAIN && tr.replay_idx)
#pragma unroll 1
      for (int j = lane; j < count; j += 32) {
        if (nrep + j < tr.replay_cap) tr.replay_idx[n * tr.replay_cap + nrep + j] = perf[j];
        else flags |= COBEL_FLAG_TRACE_OVERFLOW;
      }
    if (!PLAIN && tr.replay_len && lane == 0) {
      if (ncalls < tr.replay_calls_cap) tr.replay_len[n * tr.replay_calls_cap + ncalls] = count;
      else flags |= COBEL_FLAG_TRACE_OVERFLOW;
    }
    nrep += count;
    ++ncalls;
    __syncwarp();
  };

  // Launch phases with a single (inlined) replay site: stage 0 = end-of-trial replay of the previous trial
  // (agent/pma.py:248-256), stage 1 = [reset] + start-of-trial replay (206-213) + online steps.
  const int bw = p.sr_band;
  const double* nscr = p.need_scratch + (size_t)n * S;
  if (bulk) mbar_wait(bar, 0);                                  // Q and M.rewards have landed
  int trial = ph.trial_first, ntr = ph.n_trials;
  int s = ph.init_carry ? 0 : (int)carry[4];
  bool reset = ph.reset != 0;
  for (int stage = (ph.end_replay && do_replay) ? 0 : 1;;) {
    if (stage == 0) {
      // need = SR[last] for a trial that ended in a terminal state, else the stationary distribution
      replay((ph.scratch_need || c_last < 0) ? nscr : SRg + (size_t)c_last * S);
      stage = 1;
      continue;
    }
    if (reset) {
      win.ensure(2, lane);
      s = __ldg(p.world.starts + draw_integer(win.next(), K));
    }
    if (ntr == 0) break;
    if (do_replay)                                                           // awake replay, need = SR[start]
      replay(ph.scratch_need == 2 ? nscr + (size_t)p.n_agents * S : ph.scratch_need ? nscr : SRg + (size_t)s * S);
    double treward = 0.0;
    int step = 0, last = -1;
    for (;; ++step) {
      win.ensure(2, lane);
      // T[s] is updated at the end of the step (M.store): issue its HBM loads now, behind the action selection
      double trow[kTrow];                              // at most kTrow entries per lane
#pragma unroll
      for (int x = 0; x < kTrow; ++x) { const int j = lane + 32 * x; trow[x] = (learn && j < S) ? Tg[(size_t)s * S + j] : 0.0; }
      double row[A];
      load_row<A>(Q + s * A, row);
      const double ua = win.next();
      const int a = (PLAIN || useA) ? select_action_tab<A>(row, mbits[s], tabA, ua)
                                    : select_action_warp<A, kPol>(row, mbits[s], pt, ua, lane);
      const int s2 = (!PLAIN && p.world.tp_off) ? stochastic_successor(p.world, s * A + a, win.next()) : __ldg(p.world.succ + s * A + a);
      const double r = __ldg(p.world.reward + s2);
      const int end = __ldg(p.world.terminal + s2);
      const int nt = 1 - end;
      if (bw >= 0 && abs(s2 - s) > bw) flags |= COBEL_FLAG_BAND_VIOLATION;
      if (!PLAIN && tr.step_sa && lane == 0) {
        if (nsteps < tr.step_cap) { tr.step_sa[n * tr.step_cap + nsteps] = s * A + a; if (tr.step_next) tr.step_next[n * tr.step_cap + nsteps] = s2; }
        else flags |= COBEL_FLAG_TRACE_OVERFLOW;
      }
      ++nsteps;
      if (learn) {
        // PMA.update_q([experience]) (agent/pma.py:319-353), then M.store (memory/pma.py:148-166)
        double row2[A];
        load_row<A>(Q + s2 * A, row2);
        const double fv = xmul(row_max<A>(row2), nt ? 1.0 : 0.0);
        const double rr = xadd(0.0, xmul(r, 1.0));
        double td = xadd(rr, xmul(fv, gamma));
        const double q = Q[s * A + a];
        td = xsub(td, q);
        const double qn = xadd(q, xmul(lr, td));
        if (!PLAIN && tr.step_td && lane == 0) {       // the step's slot of step_sa
          if (nsteps <= tr.step_cap) tr.step_td[n * tr.step_cap + nsteps - 1] = td;
          else flags |= COBEL_FLAG_TRACE_OVERFLOW;
        }
        const double m0 = Mr[s * A + a];
        const double m1 = xadd(m0, xmul(mlr, xsub(r, m0)));
#pragma unroll
        for (int x = 0; x < kTrow; ++x) {              // T[s] += lr_T * (onehot(s') - T[s]), memory/pma.py:162-165
          const int j = lane + 32 * x;
          if (j < S) Tg[(size_t)s * S + j] = xadd(trow[x], xmul(p.lr_T, xsub(j == s2 ? 1.0 : 0.0, trow[x])));
        }
        __syncwarp();
        if (lane == 0) {
          Q[s * A + a] = qn;
          Mr[s * A + a] = m1;
          Pk[s * A + a] = (uint16_t)((Pk[s * A + a] & kUm) | s2 | (nt << 15));
        }
        __syncwarp();
      }
      s = s2;
      treward = xadd(treward, r);
      if (end) last = s2;
      if (end || step + 1 == p.steps) break;
    }
    if (lane == 0) {
      tr.trial_steps[n * p.trials + trial] = step;
      tr.trial_reward[n * p.trials + trial] = treward;
    }
    c_last = last;
    ++trial; --ntr;
    reset = true;                                        // further trials of this launch (no replays) reset themselves
    if (ntr == 0) break;
  }

  __syncwarp();
  if (learn) {
    // Stage-out: a launch without online steps (an end-of-trial replay) has changed Q only
    const bool stepped = ph.n_trials > 0;
    if (bulk) {
      fence_async_smem();                                       // the bulk stores read what the lanes wrote
      __syncwarp();
      if (lane == 0) {
        bulk_store_issue(p.Q + g0, Q, (unsigned)N * 8u);
        if (stepped) bulk_store_issue(p.Mr + g0, Mr, (unsigned)N * 8u);
        bulk_commit();
      }
    } else {
#pragma unroll 1
      for (int e = lane; e < N; e += 32) { p.Q[g0 + e] = Q[e]; if (stepped) p.Mr[g0 + e] = Mr[e]; }
    }
    if (stepped) {
#pragma unroll 4
      for (int e = lane; e < N; e += 32) {
        p.Ms[g0 + e] = Pk[e] & kSt;
        p.Mt[g0 + e] = Pk[e] >> 15;
      }
    }
  }
  flags = __reduce_or_sync(kFull, flags);
  if (lane == 0) {
    p.stream.draw_count[n] = (int64_t)win.position();
    carry[0] = c_last; carry[1] = nsteps; carry[2] = nrep; carry[3] = ncalls; carry[4] = s;
    tr.n_steps[n] += nsteps - nsteps0;
    tr.n_replay[n] += nrep - nrep0;
    if (tr.flags && flags) tr.flags[n] |= flags;
    if (p.min_gap && gap_num < 1e300) p.min_gap[n] = fmin(p.min_gap[n], gap_num / gap_den);
    if (learn && bulk) bulk_store_wait();                       // shared memory must outlive the bulk stores
  }
}

// Shared memory of the main kernel (kMainWarps agents per CTA)
template <int A>
int main_smem(int S, size_t& bytes) {
  bytes = (size_t)kMainWarps * MainSmem(S, A).bytes;
  COBEL_REQUIRE(bytes <= kMaxSmem, COBEL_EUNSUPPORTED, "PMA: %d states x %d actions do not fit in shared memory", S, A);
  return COBEL_OK;
}

// The dense update_sr kernel for S states (register tile 7 up to 112 states, else 10) and its shared memory
auto sr_kernel_for(int S, size_t& bytes) {
  const int tile = S <= 7 * 16 ? 7 : 10;
  bytes = (size_t)(4 * (tile * 16 + 2) + ((S + 1) & ~1) + S * S) * 8;
  return tile == 7 ? pma_sr_kernel<7> : pma_sr_kernel<10>;
}

// The final SR refresh of a banded call (the narrowest register window BW >= sr_band) and its shared memory
auto sr_band_kernel_for(int S, int sr_band, size_t& bytes) {
  static const struct { int bw; void (*kernel)(CobelPMAParams); } kLadder[] = {
      {4, pma_sr_band_kernel<4>}, {6, pma_sr_band_kernel<6>}, {8, pma_sr_band_kernel<8>}, {10, pma_sr_band_kernel<10>},
      {12, pma_sr_band_kernel<12>}, {16, pma_sr_band_kernel<16>}, {24, pma_sr_band_kernel<24>}, {32, pma_sr_band_kernel<32>}};
  int i = 0;
  while (i < 7 && kLadder[i].bw < sr_band) ++i;
  bytes = (size_t)S * (2 * kLadder[i].bw + 2) * 8;
  return kLadder[i].kernel;
}

// The tie-pattern policy tables of a call (A <= 4, n_tab > 0)
template <int A>
int policy_tables(const CobelPMAParams& p, cudaStream_t st) {
  if constexpr (A <= 4) {
    if (p.n_tab > 0)
      return launch_kernel(pma_policy_table_kernel<A>, (unsigned)p.n_tab + 1, 256, 0, st, p.tab_kind, p.tab_param, p.tab_scratch);
  }
  return COBEL_OK;
}

// The size errors shared by train() / test() and the stand-alone replay
constexpr const char* kSizeLimit = "PMA kernels support at most 512 states and 2048 one-step backups, got %d states x %d actions";
constexpr const char* kBandRequired = "PMA: more than 160 states need the banded update_sr (sr_band >= 0; the dense S x S "
                                      "eliminations are register-tiled for S <= 160), got %d states";
constexpr const char* kRefreshTooLarge = "PMA: the final SR refresh of %d states at half band %d needs %zu bytes of shared "
                                         "memory (at most %d); beyond 160 states there is no dense update_sr to fall back on";

template <int A>
int run(const CobelPMAParams& p, cudaStream_t st) {
  const int S = p.world.n_states;
  COBEL_REQUIRE(S <= 512 && S * A <= 2048, COBEL_EUNSUPPORTED, kSizeLimit, S, A);
  const bool big = S > 160 || S * A > 1024;             // pma_main_kernel<A, false, BIG>
  size_t sm_main, sm_sr;
  if (int rc = main_smem<A>(S, sm_main)) return rc;
  COBEL_REQUIRE(p.n_tab == 0 || (p.tab_kind && p.tab_param && p.tab_scratch), COBEL_EINVAL,
                "n_tab > 0 needs tab_kind, tab_param and tab_scratch[n_tab, COBEL_PMA_TAB_DOUBLES(A)]");
  const bool plain = !big && p.n_tab > 0 && A <= 4 && p.policy.kind == COBEL_POLICY_EPS_GREEDY &&
                     p.mem_policy.kind == COBEL_POLICY_EPS_GREEDY && p.learn && !p.no_replay && !p.options &&
                     !p.world.tp_off && !p.trace.step_sa && !p.trace.step_td && !p.trace.replay_idx && !p.trace.replay_len &&
                     !p.stream.user_stream;
  const bool do_replay = p.learn && !p.no_replay;
  const bool band = do_replay && p.sr_band >= 0;
  COBEL_REQUIRE(!big || !do_replay || band, COBEL_EUNSUPPORTED, kBandRequired, S);
  const auto sr_kernel = sr_kernel_for(S, sm_sr);
  // every size is checked before the first launch: a call that cannot finish leaves Q, T and the stream untouched
  size_t sm_band = 0;
  const auto band_kernel = band ? sr_band_kernel_for(S, p.sr_band, sm_band) : nullptr;
  COBEL_REQUIRE(!band || !big || sm_band <= kMaxSmem, COBEL_EUNSUPPORTED, kRefreshTooLarge, S, p.sr_band, sm_band, kMaxSmem);
  auto main_kernel = big ? pma_main_kernel<A, false, true> : pma_main_kernel<A, false>;
  if constexpr (A <= 4) {
    if (plain) main_kernel = pma_main_kernel<A, true>;
  }
  const unsigned grid_main = (unsigned)((p.n_agents + kMainWarps - 1) / kMainWarps);
  auto main_launch = [&](MainPhase ph) { return launch_kernel(main_kernel, grid_main, kMainWarps * 32, sm_main, st, p, ph); };
  auto sr_launch = [&](int final_only) { return launch_kernel(sr_kernel, (unsigned)p.n_agents, kThreads, sm_sr, st, p, final_only); };
  int rc = policy_tables<A>(p, st);
  if (rc) return rc;
  // MainPhase{init_carry, end_replay, reset, n_trials, trial_first, scratch_need}
  if (!do_replay) return main_launch(MainPhase{1, 0, 1, p.trials, 0, 0});      // no replay: all trials in one launch
  if (band) {
    // banded update_sr, its own kernels (one warp per agent, full occupancy) between the launches of the main kernel:
    //   main(reset, start replay from the caller's SR, steps of trial 0)
    //   trial t: factor(update_sr; need of the end replay) -> main(end replay t, reset t+1)
    //            -> solve(need = SR[start]) -> main(start replay, steps of trial t+1)
    //   (a world with ONE starting state: factor also solves SR[start], and the two main launches are one)
    // and SR = inv(I - gamma T) once, densely, from the last factors
    const int warps = band_warps(S, p.sr_band);
    const unsigned grid_band = (unsigned)((p.n_agents + warps - 1) / warps);
    const size_t sm_bandk = (size_t)warps * BandSmem(S, p.sr_band).bytes;
    const auto factor_kernel = warps == kBandWarps ? pma_band_factor_kernel<kBandWarps> : pma_band_factor_kernel<kBandWarpsWide>;
    const auto solve_kernel = warps == kBandWarps ? pma_band_solve_kernel<kBandWarps> : pma_band_solve_kernel<kBandWarpsWide>;
    if (!p.band_trusted)                               // the caller's band guarantee on the initial T
      rc = launch_kernel(pma_band_check_kernel, (unsigned)p.n_agents, 256, 0, st, p);
    if (!rc) rc = main_launch(MainPhase{1, 0, 1, 1, 0, 0});
    const bool one_start = p.world.n_starts == 1;      // the start row is known before the reset draw
    for (int t = 0; t < p.trials && !rc; ++t) {
      const int more = t + 1 < p.trials ? 1 : 0;
      rc = launch_kernel(factor_kernel, grid_band, warps * 32, sm_bandk, st, p, one_start && more);
      if (rc) break;
      if (one_start) {                                 // end replay t, reset, start replay and steps of trial t + 1
        rc = main_launch(MainPhase{0, 1, more, more, t + 1, 2});
        continue;
      }
      rc = main_launch(MainPhase{0, 1, more, 0, t + 1, 1});
      if (rc || !more) break;
      rc = launch_kernel(solve_kernel, grid_band, warps * 32, sm_bandk, st, p, 4);
      if (!rc) rc = main_launch(MainPhase{0, 0, 0, 1, t + 1, 1});
    }
    if (rc) return rc;
    if (sm_band <= kMaxSmem) return launch_kernel(band_kernel, (unsigned)p.n_agents, (S + 31) & ~31, sm_band, st, p);
    return sr_launch(1);                               // (S <= 160: checked above)
  }
  // trial t: main(reset, start replay, steps) -> sr(update_sr [+ stationary]) -> main(end replay, then trial t+1)
  rc = main_launch(MainPhase{1, 0, 1, 1, 0, 0});
  for (int t = 0; t < p.trials && !rc; ++t) {
    rc = sr_launch(0);
    const int more = t + 1 < p.trials ? 1 : 0;
    if (!rc) rc = main_launch(MainPhase{0, 1, more, more, t + 1, 0});
  }
  return rc;
}

// PMAMemory.replay(Q, action_mask, batch, current_state) as a stand-alone call: the end-of-trial phase of the main kernel
// (need = SR[c] from HBM, or need_scratch for c < 0).  Up to 160 states and 1024 one-step backups the dense update_sr
// kernel supplies the refreshed SR and the stationary need; beyond that (the BIG main kernel) the banded kernels of
// train() do, so the band is required there:
//   [band check] -> update_sr: band LU [+ GTH for c < 0], then pma_sr_band_kernel refreshes SR
//                   otherwise: GTH of the agents with c < 0 only (the others read SR as stored)
//   -> main(end replay)
template <int A>
int replay_only(const CobelPMAParams& p, const int32_t* state, int update_sr, cudaStream_t st) {
  const int S = p.world.n_states;
  COBEL_REQUIRE(S <= 512 && S * A <= 2048, COBEL_EUNSUPPORTED, kSizeLimit, S, A);
  const bool big = S > 160 || S * A > 1024;
  size_t sm_main;
  if (int rc = main_smem<A>(S, sm_main)) return rc;
  const unsigned grid_main = (unsigned)((p.n_agents + kMainWarps - 1) / kMainWarps);
  const MainPhase end_replay{0, 1, 0, 0, 0, 0};
  if (!big) {
    size_t sm_sr;
    const auto sr_kernel = sr_kernel_for(S, sm_sr);
    if (int rc = policy_tables<A>(p, st)) return rc;
    if (int rc = cobel_set_carry(p.carry, 8, state, p.n_agents, st)) return rc;
    // M.update_sr() and / or the stationary need of the agents whose current state is None
    if (int rc = launch_kernel(sr_kernel, (unsigned)p.n_agents, kThreads, sm_sr, st, p, update_sr ? 0 : 2)) return rc;
    return launch_kernel(pma_main_kernel<A, false>, grid_main, kMainWarps * 32, sm_main, st, p, end_replay);
  }
  // every size is checked before the first launch, as in run<A>
  COBEL_REQUIRE(p.sr_band >= 0, COBEL_EUNSUPPORTED, kBandRequired, S);
  COBEL_REQUIRE(p.sr_band <= 31 && p.band_scratch, COBEL_EINVAL,
                "sr_band must be < 0 (dense update_sr) or 0..31 with band_scratch[N, S*(2*sr_band+1)]");
  size_t sm_band;
  const auto band_kernel = sr_band_kernel_for(S, p.sr_band, sm_band);
  COBEL_REQUIRE(!update_sr || sm_band <= kMaxSmem, COBEL_EUNSUPPORTED, kRefreshTooLarge, S, p.sr_band, sm_band, kMaxSmem);
  const int warps = band_warps(S, p.sr_band);
  const unsigned grid_band = (unsigned)((p.n_agents + warps - 1) / warps);
  const size_t sm_bandk = (size_t)warps * BandSmem(S, p.sr_band).bytes;
  int rc = policy_tables<A>(p, st);
  if (!rc) rc = cobel_set_carry(p.carry, 8, state, p.n_agents, st);
  if (!rc && !p.band_trusted) rc = launch_kernel(pma_band_check_kernel, (unsigned)p.n_agents, 256, 0, st, p);
  if (rc) return rc;
  if (update_sr) {
    const auto factor_kernel = warps == kBandWarps ? pma_band_factor_kernel<kBandWarps> : pma_band_factor_kernel<kBandWarpsWide>;
    rc = launch_kernel(factor_kernel, grid_band, warps * 32, sm_bandk, st, p, 0);
    if (!rc) rc = launch_kernel(band_kernel, (unsigned)p.n_agents, (S + 31) & ~31, sm_band, st, p);
  } else {
    const auto gth_kernel = warps == kBandWarps ? pma_band_stationary_kernel<kBandWarps> : pma_band_stationary_kernel<kBandWarpsWide>;
    rc = launch_kernel(gth_kernel, grid_band, warps * 32, sm_bandk, st, p);
  }
  if (!rc) rc = launch_kernel(pma_main_kernel<A, false, true>, grid_main, kMainWarps * 32, sm_main, st, p, end_replay);
  return rc;
}

}  // namespace

extern "C" int cobel_pma_run(const CobelPMAParams* pp, void* stream) {
  COBEL_REQUIRE(pp != nullptr, COBEL_EINVAL, "null params");
  const CobelPMAParams& p = *pp;
  int rc = cobel_validate_common(p.n_agents, p.world, p.stream, p.policy, p.trace, p.trials, p.steps);
  if (rc) return rc;
  COBEL_REQUIRE(p.Q && p.Mr && p.Ms && p.Mt && p.T && p.SR && p.update_mask && p.lr && p.gamma && p.mem_lr && p.lr_q &&
                p.gamma_q && p.gamma_sr && p.pow_gamma_sr && p.pow_gamma_q && p.mem_policy.param && p.carry &&
                p.need_scratch, COBEL_EINVAL, "agent tables missing");
  COBEL_REQUIRE(p.mem_policy.kind >= 0 && p.mem_policy.kind <= 2, COBEL_EINVAL, "bad memory policy");
  COBEL_REQUIRE(p.batch >= 0 && p.batch <= kMaxSeq, COBEL_EUNSUPPORTED, "PMA replay batch must be in 0..%d", kMaxSeq);
  COBEL_REQUIRE(p.sr_band < 0 || (p.sr_band <= 31 && p.band_scratch), COBEL_EINVAL,
                "sr_band must be < 0 (dense update_sr) or 0..31 with band_scratch[N, S*(2*sr_band+1)]");
  if ((rc = cobel_validate_replay_td(p.trace))) return rc;
  if (p.trials == 0) return COBEL_OK;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  COBEL_DISPATCH_A(p.world.n_actions, return run<A>(p, st));
}

extern "C" int cobel_pma_replay(const CobelPMAParams* pp, const int32_t* state, int update_sr, void* stream) {
  COBEL_REQUIRE(pp != nullptr && state != nullptr, COBEL_EINVAL, "null params");
  CobelPMAParams p = *pp;
  p.trace.replay_td = nullptr;                         // recorded by the fused train() only
  COBEL_REQUIRE(p.n_agents > 0 && p.stream.draw_count && p.trace.n_steps && p.trace.n_replay, COBEL_EINVAL, "stream / trace missing");
  COBEL_REQUIRE(p.Q && p.Mr && p.Ms && p.Mt && p.T && p.SR && p.update_mask && p.lr && p.gamma && p.mem_lr && p.lr_q &&
                p.gamma_q && p.gamma_sr && p.pow_gamma_sr && p.pow_gamma_q && p.mem_policy.param && p.policy.param && p.carry &&
                p.need_scratch, COBEL_EINVAL, "agent tables missing");
  COBEL_REQUIRE(p.mem_policy.kind >= 0 && p.mem_policy.kind <= 2, COBEL_EINVAL, "bad memory policy");
  COBEL_REQUIRE(p.batch >= 0 && p.batch <= kMaxSeq, COBEL_EUNSUPPORTED, "PMA replay batch must be in 0..%d", kMaxSeq);
  COBEL_REQUIRE(p.learn && !p.no_replay, COBEL_EINVAL, "cobel_pma_replay needs learn = 1 and no_replay = 0");
  COBEL_REQUIRE(p.n_tab == 0 || (p.tab_kind && p.tab_param && p.tab_scratch), COBEL_EINVAL, "policy tables incomplete");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  COBEL_DISPATCH_A(p.world.n_actions, return replay_only<A>(p, state, update_sr, st));
}
