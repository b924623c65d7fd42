// sr.cu -- K3: SR.train()/test() (tabular successor-representation agent) for N independent
// agents in one launch.
//
// Reference: agent/sr.py:142-308.  Per step
//   Q[a] = np.sum(SR * rewards, axis=1)[m(s,a)]  with m = the learned one-hot transition model
//          (sr.py:288-308; only the A modelled-successor rows are evaluated here, each as the
//          same NumPy pairwise sum -- SURVEY.md Appendix A.3/A.5),
//   action selection, environment step,
//   rewards[s'] += (r - rewards[s']) * lr;  model[s,a] = s'                      (sr.py:272-274)
//   td = e_s + gamma * (SR[s'] if non-terminal else e_s') - SR[s];  SR[s] += lr * td   (276-284)
//
// Mapping: one CTA per agent, threads parallel over the S columns of a row.  SR stays in HBM
// (S*S*8 bytes per agent: 5 KB at 5x5, 1.28 MB at 20x20) and is streamed through L1/L2 with
// coalesced fp64 row accesses: A+2 row reads and one row write per step (8S(A+4) algorithmic
// bytes); rewards / model / Q scratch live in shared memory.
#include "warp_agent.cuh"
#include "tma.cuh"

namespace {

constexpr int kMaxLeaves = 64;     // pairwise-sum leaves of <=128 elements: S <= 8192

// NumPy's pairwise summation (DOUBLE_add reduce) as a plan: leaves of 8..128 elements are summed
// with 8 strided accumulators + a sequential tail; leaf results are combined by the recursion
// `sum(n) = sum(first n2) + sum(rest)`, n2 = n/2 - (n/2)%8, flattened here in post-order.
struct PairwisePlan {
  int n, nl, nc;
  int start[kMaxLeaves + 1];
  short left[kMaxLeaves], right[kMaxLeaves];
};

int plan_rec(PairwisePlan& pl, int lo, int n) {
  if (n <= 128) {
    if (pl.nl >= kMaxLeaves) return -1;
    pl.start[pl.nl] = lo;
    pl.start[pl.nl + 1] = lo + n;
    return pl.nl++;
  }
  int n2 = n / 2;
  n2 -= n2 % 8;
  const int l = plan_rec(pl, lo, n2);
  const int r = plan_rec(pl, lo + n2, n - n2);
  if (l < 0 || r < 0) return -1;
  pl.left[pl.nc] = (short)l; pl.right[pl.nc] = (short)r;
  ++pl.nc;
  return l;              // the sum of the subtree is accumulated into its left-most leaf slot
}

bool make_plan(PairwisePlan& pl, int n) {
  pl.n = n; pl.nl = 0; pl.nc = 0;
  return plan_rec(pl, 0, n) >= 0;
}

struct SRSmem {
  int rew, prod, acc, leaf, q, model, bytes;
  __host__ __device__ SRSmem(int S, int A, int nl) {
    rew = 0;
    prod = rew + S * 8;
    acc = prod + A * S * 8;
    leaf = acc + A * nl * 8 * 8;
    q = leaf + A * nl * 8;
    model = q + A * 8;
    bytes = (model + S * A * 4 + 15) & ~15;
  }
};

template <int A>
__global__ void __launch_bounds__(256) sr_kernel(const __grid_constant__ CobelSRParams p, const __grid_constant__ PairwisePlan pl) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, K = p.world.n_starts;
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31;
  const int64_t n = blockIdx.x;
  const SRSmem so(S, A, pl.nl);
  double* rew = reinterpret_cast<double*>(smem + so.rew);
  double* prod = reinterpret_cast<double*>(smem + so.prod);      // [A][S] products SR[m_a, j] * rew[j]
  double* acc = reinterpret_cast<double*>(smem + so.acc);        // [A][nl][8]
  double* leaf = reinterpret_cast<double*>(smem + so.leaf);      // [A][nl]
  double* qv = reinterpret_cast<double*>(smem + so.q);           // [A]
  int32_t* model = reinterpret_cast<int32_t*>(smem + so.model);  // [S][A] modelled successor

  double* SR = p.SR + (size_t)n * S * S;
  for (int e = tid; e < S; e += T) rew[e] = p.rewards[(size_t)n * S + e];
  for (int e = tid; e < S * A; e += T) model[e] = p.model[(size_t)n * S * A + e];
  __syncthreads();

  DrawWindow win; win.init(p.stream, n, (uint64_t)p.stream.draw_count[n]);
  const double lr = p.lr[n], gamma = p.gamma[n];
  PolicyTab pt; pt.init(p.policy.kind, p.policy.param[n], lane);
  const uint8_t* amask = p.action_mask ? p.action_mask + n * p.mask_agent_stride : nullptr;
  const bool learn = p.learn != 0;
  const CobelTrace& tr = p.trace;
  int64_t nsteps = 0;
  int flags = 0;
  const int nl = pl.nl;

  for (int trial = 0; trial < p.trials; ++trial) {
    win.ensure(2, lane);
    int s = __ldg(p.world.starts + draw_integer(win.next(), K));
    double treward = 0.0;
    int step = 0;
    for (;; ++step) {
      // ---- retrieve_q: A row dots in NumPy's pairwise order --------------------------------
      for (int e = tid; e < A * S; e += T) {
        const int a = e / S, j = e - a * S;
        prod[e] = xmul(SR[(size_t)model[s * A + a] * S + j], rew[j]);
      }
      __syncthreads();
      for (int t = tid; t < A * nl * 8; t += T) {          // 8 strided accumulators per leaf
        const int a = t / (nl * 8), l = (t / 8) % nl, k = t & 7;
        const int lo = pl.start[l], len = pl.start[l + 1] - lo;
        const double* x = prod + a * S + lo;
        double r = 0.0;
        if (len >= 8) {
          r = x[k];
          for (int i = 8 + k; i < len - (len & 7); i += 8) r = xadd(r, x[i]);
        }
        acc[t] = r;
      }
      __syncthreads();
      for (int t = tid; t < A * nl; t += T) {              // combine + sequential tail
        const int a = t / nl, l = t - a * nl;
        const int lo = pl.start[l], len = pl.start[l + 1] - lo;
        const double* x = prod + a * S + lo;
        const double* r = acc + t * 8;
        double res;
        int i;
        if (len < 8) {
          res = 0.0; i = 0;
        } else {
          res = xadd(xadd(xadd(r[0], r[1]), xadd(r[2], r[3])), xadd(xadd(r[4], r[5]), xadd(r[6], r[7])));
          i = len - (len & 7);
        }
        for (; i < len; ++i) res = xadd(res, x[i]);
        leaf[t] = res;
      }
      __syncthreads();
      if (tid < A) {                                       // recursion over the leaves, post-order
        double* L = leaf + tid * nl;
        for (int c = 0; c < pl.nc; ++c) L[pl.left[c]] = xadd(L[pl.left[c]], L[pl.right[c]]);
        qv[tid] = L[0];
      }
      __syncthreads();
      // ---- action selection and environment step: every warp computes the same (warp-uniform)
      // result, which keeps all warps' stream windows in lock-step without a broadcast ---------
      win.ensure(2, lane);
      double row[A];
#pragma unroll
      for (int x = 0; x < A; ++x) row[x] = qv[x];
      uint32_t mask = (1u << A) - 1u;
      if (amask) {
        mask = 0;
#pragma unroll
        for (int x = 0; x < A; ++x) mask |= (amask[s * A + x] ? 1u : 0u) << x;
      }
      const int a = select_action_warp<A>(row, mask, pt, win.next(), lane);
      const int s2 = p.world.tp_off ? stochastic_successor(p.world, s * A + a, win.next()) : __ldg(p.world.succ + s * A + a);
      const double r = __ldg(p.world.reward + s2);
      const int end = __ldg(p.world.terminal + s2);
      if (tr.step_sa && tid == 0) {
        if (nsteps < tr.step_cap) { tr.step_sa[n * tr.step_cap + nsteps] = s * A + a; if (tr.step_next) tr.step_next[n * tr.step_cap + nsteps] = s2; }
        else flags |= COBEL_FLAG_TRACE_OVERFLOW;
      }
      ++nsteps;
      if (learn) {
        // ---- SR.update (sr.py:255-286): every thread owns columns j = tid, tid+T, ... ----------
        const double* rs = SR + (size_t)s * S;
        const double* rs2 = SR + (size_t)s2 * S;
        double* wr = SR + (size_t)s * S;
        for (int j = tid; j < S; j += T) {
          const double old = rs[j];
          const double x = end ? (j == s2 ? 1.0 : 0.0) : rs2[j];
          double td = xadd(j == s ? 1.0 : 0.0, xmul(gamma, x));
          td = xsub(td, old);
          // all reads of row s (as SR[s] and, when s2 == s, as SR[s2]) precede this write of column j
          wr[j] = xadd(old, xmul(lr, td));
        }
        if (tid == 0) {
          const double r0 = rew[s2];
          rew[s2] = xadd(r0, xmul(xsub(r, r0), lr));
          model[s * A + a] = s2;
        }
        __syncthreads();
      }
      s = s2;
      treward = xadd(treward, r);
      if (end || step + 1 == p.steps) break;
    }
    if (tid == 0) {
      tr.trial_steps[n * p.trials + trial] = step;
      tr.trial_reward[n * p.trials + trial] = treward;
    }
  }

  __syncthreads();
  if (learn) {
    for (int e = tid; e < S; e += T) p.rewards[(size_t)n * S + e] = rew[e];
    for (int e = tid; e < S * A; e += T) p.model[(size_t)n * S * A + e] = model[e];
  }
  if (tid == 0) {
    p.stream.draw_count[n] = (int64_t)win.position();
    tr.n_steps[n] += nsteps;
    if (tr.flags && flags) tr.flags[n] |= flags;
  }
}

// ---------------------------------------------------------------------------
// sr_tma_kernel: the same agent, rows of SR streamed by the TMA (bulk asynchronous copies, cp.async.bulk + mbarrier).
//
// A step reads A + 2 rows of the agent's S x S matrix in HBM/L2 and writes one.  sr_kernel fetches them with
// per-thread loads inside the passes that consume them (5 block barriers and 5600 warp-instructions per step at
// 20x20, profiles/r2_sr_dense.txt).  Here one elected thread issues whole-row bulk copies into shared memory and the
// passes read shared memory only:
//   * the A successor rows of the NEXT step are requested as soon as the next state is known, i.e. they fly
//     while the current step's row update runs (into the same buffer: the pairwise sums of the current step are
//     done by then; a row that is being rewritten is requested after its write-back has completed);
//   * the updated row goes back with one bulk store;
//   * the products SR[m, j] * rewards[j] are formed inside the pairwise-sum chains (no product pass), the leaf
//     combine, the recursion over the leaves, action selection and the environment step run in warp 0 only.
// Rows must be 16-byte multiples (S even); odd S and state spaces whose rows do not fit in shared memory take
// sr_kernel.
// ---------------------------------------------------------------------------
struct SRTmaSmem {
  int rew, rows, urow, acc, leaf, q, model, bars, bytes;
  __host__ __device__ SRTmaSmem(int S, int A, int nl) {
    rew = 0;
    rows = rew + S * 8;                  // [A][S] successor rows of the current step, then of the next one
    urow = rows + A * S * 8;             // [2][S] rows s and s' of the update
    acc = urow + 2 * S * 8;              // [A][nl][8]
    leaf = acc + A * nl * 8 * 8;         // [A][nl]
    q = leaf + A * nl * 8;
    bars = q + ((A + 1) & ~1) * 8;       // 2 mbarriers
    model = bars + 32;
    bytes = (model + S * A * 4 + 15) & ~15;
  }
};

struct SRStepShared { int a, s2, end, last; double r; };

template <int A>
__global__ void __launch_bounds__(128) sr_tma_kernel(const __grid_constant__ CobelSRParams p, const __grid_constant__ PairwisePlan pl) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ SRStepShared sh;
  const int S = p.world.n_states, K = p.world.n_starts;
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int64_t n = blockIdx.x;
  const int nl = pl.nl;
  const SRTmaSmem so(S, A, nl);
  double* rew = reinterpret_cast<double*>(smem + so.rew);
  double* rows = reinterpret_cast<double*>(smem + so.rows);
  double* urow = reinterpret_cast<double*>(smem + so.urow);
  double* acc = reinterpret_cast<double*>(smem + so.acc);
  double* leaf = reinterpret_cast<double*>(smem + so.leaf);
  double* qv = reinterpret_cast<double*>(smem + so.q);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + so.bars);     // [0]: the successor rows; [1]: the update rows
  int32_t* model = reinterpret_cast<int32_t*>(smem + so.model);
  const unsigned row_bytes = (unsigned)S * 8u;

  double* SR = p.SR + (size_t)n * S * S;
  for (int e = tid; e < S; e += T) rew[e] = p.rewards[(size_t)n * S + e];
  for (int e = tid; e < S * A; e += T) model[e] = p.model[(size_t)n * S * A + e];
  if (tid == 0) {
    mbar_init(&bars[0], 1); mbar_init(&bars[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  DrawWindow win; win.init(p.stream, n, (uint64_t)p.stream.draw_count[n]);      // used by warp 0 only
  const double lr = p.lr[n], gamma = p.gamma[n];
  PolicyTab pt; pt.init(p.policy.kind, p.policy.param[n], lane);
  const uint8_t* amask = p.action_mask ? p.action_mask + n * p.mask_agent_stride : nullptr;
  const bool learn = p.learn != 0;
  const CobelTrace& tr = p.trace;
  int64_t nsteps = 0;
  int flags = 0;
  unsigned ph_rows = 0u, ph_upd = 0u;                // phase parities (block-uniform)
  bool store_pending = false;                        // (thread 0) a write-back may still be in flight

  // (thread 0) request the A successor rows of state s; rows equal to `hold` are left out and returned as a bit
  // mask (they are being rewritten).  The row set is free as soon as the pairwise sums of the current step are
  // done, so the next step's rows land in the same buffer while the update runs.
  auto request_rows = [&](int s, int hold) -> unsigned {
    mbar_expect_tx(&bars[0], (unsigned)A * row_bytes);
    unsigned deferred = 0;
#pragma unroll
    for (int a = 0; a < A; ++a) {
      const int m = model[s * A + a];
      if (m == hold) deferred |= 1u << a;
      else bulk_load(rows + (size_t)a * S, SR + (size_t)m * S, row_bytes, &bars[0]);
    }
    return deferred;
  };

  for (int trial = 0; trial < p.trials; ++trial) {
    if (warp == 0) {
      win.ensure(2, lane);
      const int s0 = __ldg(p.world.starts + draw_integer(win.next(), K));
      if (lane == 0) {
        sh.s2 = s0;
        if (store_pending) { bulk_store_wait(); store_pending = false; }
        request_rows(s0, -1);
      }
    }
    __syncthreads();
    int s = sh.s2;
    double treward = 0.0;
    int step = 0;
    for (;; ++step) {
      // ---- retrieve_q: A row dots in NumPy's pairwise order, straight from the TMA-filled row set ------------
      mbar_wait(&bars[0], ph_rows);
      ph_rows ^= 1u;
      const double* rset = rows;
      for (int t = tid; t < A * nl * 8; t += T) {          // 8 strided accumulators per leaf
        const int a = t / (nl * 8), l = (t / 8) % nl, k = t & 7;
        const int lo = pl.start[l], len = pl.start[l + 1] - lo;
        const double* x = rset + a * S + lo;
        const double* w = rew + lo;
        double r = 0.0;
        if (len >= 8) {
          r = xmul(x[k], w[k]);
          for (int i = 8 + k; i < len - (len & 7); i += 8) r = xadd(r, xmul(x[i], w[i]));
        }
        acc[t] = r;
      }
      __syncthreads();
      if (warp == 0) {
        for (int t = lane; t < A * nl; t += 32) {          // combine + sequential tail
          const int a = t / nl, l = t - a * nl;
          const int lo = pl.start[l], len = pl.start[l + 1] - lo;
          const double* x = rset + a * S + lo;
          const double* w = rew + lo;
          const double* r = acc + t * 8;
          double res;
          int i;
          if (len < 8) {
            res = 0.0; i = 0;
          } else {
            res = xadd(xadd(xadd(r[0], r[1]), xadd(r[2], r[3])), xadd(xadd(r[4], r[5]), xadd(r[6], r[7])));
            i = len - (len & 7);
          }
          for (; i < len; ++i) res = xadd(res, xmul(x[i], w[i]));
          leaf[t] = res;
        }
        __syncwarp();
        if (lane < A) {                                     // recursion over the leaves, post-order
          double* L = leaf + lane * nl;
          for (int c = 0; c < pl.nc; ++c) L[pl.left[c]] = xadd(L[pl.left[c]], L[pl.right[c]]);
          qv[lane] = L[0];
        }
        __syncwarp();
        // ---- action selection and environment step -----------------------------------------------------
        win.ensure(2, lane);
        double row[A];
#pragma unroll
        for (int x = 0; x < A; ++x) row[x] = qv[x];
        uint32_t mask = (1u << A) - 1u;
        if (amask) {
          mask = 0;
#pragma unroll
          for (int x = 0; x < A; ++x) mask |= (amask[s * A + x] ? 1u : 0u) << x;
        }
        const int a = select_action_warp<A>(row, mask, pt, win.next(), lane);
        const int s2 = p.world.tp_off ? stochastic_successor(p.world, s * A + a, win.next()) : __ldg(p.world.succ + s * A + a);
        const double r = __ldg(p.world.reward + s2);
        const int end = __ldg(p.world.terminal + s2);
        const int last = (end || step + 1 == p.steps) ? 1 : 0;
        if (lane == 0) {
          if (tr.step_sa) {
            if (nsteps < tr.step_cap) { tr.step_sa[n * tr.step_cap + nsteps] = s * A + a; if (tr.step_next) tr.step_next[n * tr.step_cap + nsteps] = s2; }
            else flags |= COBEL_FLAG_TRACE_OVERFLOW;
          }
          sh.a = a; sh.s2 = s2; sh.end = end; sh.last = last; sh.r = r;
          unsigned deferred = 0;
          if (store_pending) { bulk_store_wait(); store_pending = false; }   // rows requested below may have been rewritten
          if (learn) {
            // rows s and s' of the update; the learned model changes before the next step's rows are chosen
            mbar_expect_tx(&bars[1], (end ? 1u : 2u) * row_bytes);
            bulk_load(urow, SR + (size_t)s * S, row_bytes, &bars[1]);
            if (!end) bulk_load(urow + S, SR + (size_t)s2 * S, row_bytes, &bars[1]);
            model[s * A + a] = s2;
          }
          if (!last) deferred = request_rows(s2, learn ? s : -1);
          sh.last |= (int)(deferred << 8);
        }
      }
      ++nsteps;
      __syncthreads();
      const int a = sh.a, s2 = sh.s2, end = sh.end, last = sh.last & 1;
      const unsigned deferred = (unsigned)sh.last >> 8;
      const double r = sh.r;
      (void)a;
      if (learn) {
        // ---- SR.update (sr.py:255-286) on the staged rows; every thread owns columns j = tid, tid+T, ... ------
        mbar_wait(&bars[1], ph_upd);
        ph_upd ^= 1u;
        for (int j = tid; j < S; j += T) {
          const double old = urow[j];
          const double x = end ? (j == s2 ? 1.0 : 0.0) : urow[S + j];
          double td = xadd(j == s ? 1.0 : 0.0, xmul(gamma, x));
          td = xsub(td, old);
          urow[j] = xadd(old, xmul(lr, td));
        }
        if (tid == 0) {
          const double r0 = rew[s2];
          rew[s2] = xadd(r0, xmul(xsub(r, r0), lr));
        }
        fence_async_smem();                                 // the bulk store below reads what the threads wrote
        __syncthreads();
        if (tid == 0) {
          bulk_store(SR + (size_t)s * S, urow, row_bytes);
          store_pending = true;
          if (deferred) {                                   // next-step rows that are this very row: after the write-back
            bulk_store_wait(); store_pending = false;
#pragma unroll
            for (int x = 0; x < A; ++x)
              if (deferred >> x & 1u) bulk_load(rows + (size_t)x * S, SR + (size_t)s * S, row_bytes, &bars[0]);
          }
        }
      }
      s = s2;
      treward = xadd(treward, r);
      if (last) break;
    }
    if (tid == 0) {
      tr.trial_steps[n * p.trials + trial] = step;
      tr.trial_reward[n * p.trials + trial] = treward;
    }
    __syncthreads();                                        // everyone has read the last step's broadcast
  }

  if (tid == 0 && store_pending) bulk_store_wait();
  __syncthreads();
  if (learn) {
    for (int e = tid; e < S; e += T) p.rewards[(size_t)n * S + e] = rew[e];
    for (int e = tid; e < S * A; e += T) p.model[(size_t)n * S * A + e] = model[e];
  }
  if (tid == 0) {
    p.stream.draw_count[n] = (int64_t)win.position();
    tr.n_steps[n] += nsteps;
    if (tr.flags && flags) tr.flags[n] |= flags;
  }
}

template <int A>
int launch(const CobelSRParams& p, cudaStream_t st) {
  const int S = p.world.n_states;
  PairwisePlan pl;
  COBEL_REQUIRE(make_plan(pl, S), COBEL_EUNSUPPORTED, "dense SR kernel supports at most %d states", kMaxLeaves * 128);
  // TMA path: rows are 16-byte multiples and both row sets fit in shared memory
  const SRTmaSmem to(S, A, pl.nl);
  if (S % 2 == 0 && to.bytes <= 200 * 1024)
    return launch_kernel(sr_tma_kernel<A>, (unsigned)p.n_agents, 128, to.bytes, st, p, pl);
  const SRSmem so(S, A, pl.nl);
  COBEL_REQUIRE(so.bytes <= kMaxSmem, COBEL_EUNSUPPORTED, "dense SR kernel: %d states need %d bytes of shared memory",
                S, so.bytes);
  const int T = S <= 32 ? 32 : S <= 64 ? 64 : S <= 256 ? 128 : 256;
  return launch_kernel(sr_kernel<A>, (unsigned)p.n_agents, T, so.bytes, st, p, pl);
}

}  // namespace

extern "C" int cobel_sr_run(const CobelSRParams* pp, void* stream) {
  COBEL_REQUIRE(pp != nullptr, COBEL_EINVAL, "null params");
  const CobelSRParams& p = *pp;
  int rc = cobel_validate_common(p.n_agents, p.world, p.stream, p.policy, p.trace, p.trials, p.steps);
  if (rc) return rc;
  COBEL_REQUIRE(p.SR && p.rewards && p.model && p.lr && p.gamma, COBEL_EINVAL, "agent tables missing");
  if (p.trials == 0) return COBEL_OK;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  COBEL_DISPATCH_A(p.world.n_actions, return launch<A>(p, st));
}
