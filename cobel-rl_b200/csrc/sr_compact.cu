// sr_compact.cu -- K3b: SR agent on very large state spaces (BASELINE.json config C5: 100x100
// gridworld, 1M agents) with a per-agent VISITED-SET COMPACTION of the successor representation.
//
// Reference: agent/sr.py:142-308 (same algorithm as sr.cu).  The reference holds SR as a dense
// S x S matrix (800 MB per agent at S = 10^4) and the one-hot transition model as S x A x S
// (3.2 GB).  Rows of never-visited states stay e_s and supp(SR[s]) is a subset of the states
// touched so far, so each agent only needs
//     visited[V]            local index -> global state (insertion order), V <= Vmax
//     SRc[V][V]             SRc[i][j] = SR[visited[i]][visited[j]]
//     rew[V], model[V][A]   learned reward / modelled successor (local index) of visited states
// and every other entry of the dense tables is implied (identity rows, self-loop model, zero
// reward).  SURVEY.md section 7.3-1.
//
// Q[a] = np.sum(SR[m(s,a), :] * rewards) must reproduce NumPy's pairwise summation over all S
// columns because the policy tests exact equality of Q-values.  Only columns with a non-zero
// learned reward contribute a non-zero product, and adding an exact zero is a no-op, so the sum
// is evaluated over those few columns in the pairwise tree determined by their GLOBAL index
// (pairwise_sparse below): bit-identical to the dense result.
//
// Mapping: one warp per agent; visited / rew / model in shared memory (1.8 KB per agent at
// Vmax = 128, 64 agents per SM), SRc in HBM (row reads / one row write per step, coalesced).
// Algorithmic bytes per step: 8V(A+4)+24 with V the current visited count (SURVEY.md 8d).
#include "warp_agent.cuh"

namespace {

constexpr int kWarpsPerCta = 4;

// NumPy pairwise sum of a length-n vector whose only non-zero entries are val[t] at sorted
// positions pos[t], t < k.  Follows DOUBLE_add's tree: n < 8 sequential; n <= 128: 8 strided
// accumulators over the first n - n%8 elements, combined ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)),
// then the tail sequentially; n > 128: sum(first n2) + sum(rest), n2 = n/2 - (n/2)%8.
__device__ __noinline__ double pairwise_sparse(const int* pos, const double* val, int k, int n_total) {
  if (k == 0) return 0.0;
  if (k == 1) return xadd(0.0, val[0]);
  struct Frame { int lo, n, phase; double left; };
  Frame st[20];
  int sp = 0, idx = 0;
  double ret = 0.0;
  st[sp++] = Frame{0, n_total, 0, 0.0};
  while (sp > 0) {
    Frame& f = st[sp - 1];
    if (f.phase == 0) {
      if (idx >= k || pos[idx] >= f.lo + f.n) { ret = 0.0; --sp; continue; }      // all-zero range
      if (f.n <= 128) {
        double res;
        if (f.n < 8) {
          res = 0.0;
          while (idx < k && pos[idx] < f.lo + f.n) res = xadd(res, val[idx++]);
        } else {
          double r[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
          const int main_end = f.lo + f.n - (f.n & 7);
          while (idx < k && pos[idx] < main_end) { const int t = (pos[idx] - f.lo) & 7; r[t] = xadd(r[t], val[idx]); ++idx; }
          res = xadd(xadd(xadd(r[0], r[1]), xadd(r[2], r[3])), xadd(xadd(r[4], r[5]), xadd(r[6], r[7])));
          while (idx < k && pos[idx] < f.lo + f.n) res = xadd(res, val[idx++]);
        }
        ret = res; --sp; continue;
      }
      int n2 = f.n / 2; n2 -= n2 % 8;
      f.phase = 1;
      st[sp++] = Frame{f.lo, n2, 0, 0.0};
    } else if (f.phase == 1) {
      int n2 = f.n / 2; n2 -= n2 % 8;
      f.left = ret; f.phase = 2;
      st[sp++] = Frame{f.lo + n2, f.n - n2, 0, 0.0};
    } else {
      ret = xadd(f.left, ret); --sp;
    }
  }
  return ret;
}

struct CompactSmem {
  int rew, pos, val, vis, model, lidx, sidx, ptab, bytes;
  __host__ __device__ CompactSmem(int Vmax, int A) {
    rew = 0;
    val = rew + Vmax * 8;              // products of one row, A rows
    pos = val + A * Vmax * 8;          // sorted global positions of the reward-carrying columns
    lidx = pos + Vmax * 4;             // their local indices (unsorted / sorted)
    sidx = lidx + Vmax * 4;
    vis = sidx + Vmax * 4;
    model = vis + Vmax * 4;
    ptab = (model + Vmax * A * 2 + 15) & ~15;
    bytes = ptab + kEpsTabDoubles * 8;   // tie-pattern CDF table of the PLAIN kernel (warp_agent.cuh)
  }
};

// PLAIN = no optional trace buffers, no action mask, deterministic world (see dynaq.cu)
template <int A, bool PLAIN>
__global__ void __launch_bounds__(kWarpsPerCta * 32) sr_compact_kernel(const __grid_constant__ CobelSRCompactParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, K = p.world.n_starts, Vmax = p.max_visited;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n = (int64_t)blockIdx.x * kWarpsPerCta + warp;
  if (n >= p.n_agents) return;
  const CompactSmem so(Vmax, A);
  unsigned char* blk = smem + (size_t)warp * so.bytes;
  double* rew = reinterpret_cast<double*>(blk + so.rew);        // [V]
  double* val = reinterpret_cast<double*>(blk + so.val);        // [A][k]
  int32_t* pos = reinterpret_cast<int32_t*>(blk + so.pos);      // [k]
  int32_t* lidx = reinterpret_cast<int32_t*>(blk + so.lidx);    // [k]
  int32_t* sidx = reinterpret_cast<int32_t*>(blk + so.sidx);    // [k]
  int32_t* vis = reinterpret_cast<int32_t*>(blk + so.vis);      // [V] local -> global
  uint16_t* model = reinterpret_cast<uint16_t*>(blk + so.model);// [V][A] local successor

  double* SRc = p.SRc + (size_t)n * Vmax * Vmax;
  int V = p.n_visited[n];
  for (int e = lane; e < V; e += 32) { rew[e] = p.rewards[(size_t)n * Vmax + e]; vis[e] = p.visited[(size_t)n * Vmax + e]; }
  for (int e = lane; e < V * A; e += 32) model[e] = (uint16_t)p.model[(size_t)n * Vmax * A + e];
  __syncwarp();

  // two draws per step: the 64-draw register window wastes nothing here (a shared-memory window measured 10 % slower)
  DrawWindowT<!PLAIN> win; win.init(p.stream, n, (uint64_t)p.stream.draw_count[n]);
  const double lr = p.lr[n], gamma = p.gamma[n];
  PolicyTab pt; pt.init(p.policy.kind, p.policy.param[n], lane);
  constexpr bool kEpsTab = PLAIN && A <= 4;
  double* ptab = reinterpret_cast<double*>(blk + so.ptab);
  if constexpr (kEpsTab) eps_cdf_table_init<A>(ptab, pt, lane);
  const bool learn = p.learn != 0;
  const CobelTrace& tr = p.trace;
  int64_t nsteps = 0;
  int flags = 0;

  // local index of a global state; a new state gets the next index with an identity row,
  // a zero column, a self-loop model and zero reward (agent/sr.py:130-136)
  auto locate = [&](int g) -> int {
    unsigned hit = 0;
    int where = -1;
    // newest entries first: a walk mostly returns to states it has just left (entries are unique: at most one hit)
    for (int e0 = (V - 1) & ~31; e0 >= 0; e0 -= 32) {
      const int e = e0 + lane;
      hit = __ballot_sync(kFull, e < V && vis[e] == g);
      if (hit) { where = e0 + __ffs(hit) - 1; break; }
    }
    if (where >= 0) return where;
    if (V >= Vmax) { flags |= COBEL_FLAG_VISITED_OVERFLOW; return Vmax - 1; }
    const int v = V;
    for (int j = lane; j <= v; j += 32) SRc[(size_t)v * Vmax + j] = j == v ? 1.0 : 0.0;
    for (int i = lane; i < v; i += 32) SRc[(size_t)i * Vmax + v] = 0.0;
    if (lane == 0) { vis[v] = g; rew[v] = 0.0; }
    if (lane < A) model[v * A + lane] = (uint16_t)v;
    ++V;
    __syncwarp();
    return v;
  };

  for (int trial = 0; trial < p.trials; ++trial) {
    win.ensure(2, lane);
    int s = __ldg(p.world.starts + draw_integer(win.next(), K));
    int ls = locate(s);
    double treward = 0.0;
    int step = 0;
    for (;; ++step) {
      // ---- retrieve_q (agent/sr.py:288-308) over the reward-carrying columns only ----------------
      int k = 0;
      for (int e0 = 0; e0 < V; e0 += 32) {
        const int e = e0 + lane;
        const bool nz = e < V && rew[e] != 0.0;
        const unsigned b = __ballot_sync(kFull, nz);
        if (nz) lidx[k + __popc(b & ((1u << lane) - 1u))] = e;
        k += __popc(b);
      }
      __syncwarp();
      // rank-sort the k columns by global index (global states are distinct, so ranks are unique)
      for (int t = lane; t < k; t += 32) {
        const int e = lidx[t], g = vis[e];
        int rank = 0;
        for (int u = 0; u < k; ++u) rank += vis[lidx[u]] < g ? 1 : 0;
        pos[rank] = g;
        sidx[rank] = e;
      }
      __syncwarp();
      for (int e = lane; e < A * k; e += 32) {       // products SR[m_a, j] * rew[j] in sorted column order
        const int a = e / k, t = e - a * k;
        const int m = model[ls * A + a], lj = sidx[t];
        val[a * Vmax + t] = xmul(SRc[(size_t)m * Vmax + lj], rew[lj]);
      }
      __syncwarp();
      double qa = 0.0;
      if (lane < A) qa = pairwise_sparse(pos, val + lane * Vmax, k, S);
      double row[A];
#pragma unroll
      for (int a = 0; a < A; ++a) row[a] = shfl_f64(qa, a);
      // ---- action selection, environment step ----------------------------------------------------
      win.ensure(2, lane);
      uint32_t mask = (1u << A) - 1u;
      if (!PLAIN && p.action_mask) {
        mask = 0;
#pragma unroll
        for (int a = 0; a < A; ++a) mask |= (p.action_mask[(size_t)s * A + a] ? 1u : 0u) << a;
      }
      int a;
      if constexpr (kEpsTab) a = select_action_eps_tab<A>(row, ptab, win.next(), lane);
      else a = select_action_warp<A, PLAIN ? COBEL_POLICY_EPS_GREEDY : -1>(row, mask, pt, win.next(), lane);
      const int s2 = (!PLAIN && p.world.tp_off) ? stochastic_successor(p.world, s * A + a, win.next()) : __ldg(p.world.succ + (size_t)s * A + a);
      const double r = __ldg(p.world.reward + s2);
      const int end = __ldg(p.world.terminal + s2);
      if (!PLAIN && tr.step_sa && lane == 0) {
        if (nsteps < tr.step_cap) { tr.step_sa[n * tr.step_cap + nsteps] = s * A + a; if (tr.step_next) tr.step_next[n * tr.step_cap + nsteps] = s2; }
        else flags |= COBEL_FLAG_TRACE_OVERFLOW;
      }
      ++nsteps;
      int ls2 = ls;
      if (learn) {
        ls2 = locate(s2);
        // ---- SR.update (agent/sr.py:255-286) on the visited columns -------------------------------
        const double* rs = SRc + (size_t)ls * Vmax;
        const double* rs2 = SRc + (size_t)ls2 * Vmax;
        double* wr = SRc + (size_t)ls * Vmax;
        for (int j = lane; j < V; j += 32) {
          const double old = rs[j];
          const double x = end ? (j == ls2 ? 1.0 : 0.0) : rs2[j];
          double td = xadd(j == ls ? 1.0 : 0.0, xmul(gamma, x));
          td = xsub(td, old);
          wr[j] = xadd(old, xmul(lr, td));
        }
        if (lane == 0) {
          const double r0 = rew[ls2];
          rew[ls2] = xadd(r0, xmul(xsub(r, r0), lr));
          model[ls * A + a] = (uint16_t)ls2;
        }
        __syncwarp();
      } else if (!end && step + 1 != p.steps) {
        ls2 = locate(s2);                            // test(): still needs the local index to act from s2
      }
      s = s2; ls = ls2;
      treward = xadd(treward, r);
      if (end || step + 1 == p.steps) break;
    }
    if (lane == 0) {
      tr.trial_steps[n * p.trials + trial] = step;
      tr.trial_reward[n * p.trials + trial] = treward;
    }
  }

  __syncwarp();
  for (int e = lane; e < V; e += 32) { p.rewards[(size_t)n * Vmax + e] = rew[e]; p.visited[(size_t)n * Vmax + e] = vis[e]; }
  for (int e = lane; e < V * A; e += 32) p.model[(size_t)n * Vmax * A + e] = model[e];
  flags = __reduce_or_sync(kFull, flags);
  if (lane == 0) {
    p.n_visited[n] = V;
    p.stream.draw_count[n] = (int64_t)win.position();
    tr.n_steps[n] += nsteps;
    if (tr.flags && flags) tr.flags[n] |= flags;
  }
}

template <int A>
int launch(const CobelSRCompactParams& p, cudaStream_t st) {
  const CompactSmem so(p.max_visited, A);
  const size_t sm = (size_t)kWarpsPerCta * so.bytes;
  COBEL_REQUIRE(sm <= kMaxSmem, COBEL_EUNSUPPORTED, "max_visited %d does not fit in shared memory", p.max_visited);
  const bool plain = !p.action_mask && !p.world.tp_off && !p.trace.step_sa && p.policy.kind == COBEL_POLICY_EPS_GREEDY &&
                     !p.stream.user_stream;
  return launch_kernel(plain ? sr_compact_kernel<A, true> : sr_compact_kernel<A, false>,
                       (unsigned)((p.n_agents + kWarpsPerCta - 1) / kWarpsPerCta), kWarpsPerCta * 32, sm, st, p);
}

}  // namespace

extern "C" int cobel_sr_compact_run(const CobelSRCompactParams* pp, void* stream) {
  COBEL_REQUIRE(pp != nullptr, COBEL_EINVAL, "null params");
  const CobelSRCompactParams& p = *pp;
  int rc = cobel_validate_common(p.n_agents, p.world, p.stream, p.policy, p.trace, p.trials, p.steps);
  if (rc) return rc;
  COBEL_REQUIRE(p.SRc && p.rewards && p.model && p.visited && p.n_visited && p.lr && p.gamma, COBEL_EINVAL,
                "agent tables missing");
  COBEL_REQUIRE(p.max_visited >= 2 && p.max_visited <= 65535, COBEL_EINVAL, "max_visited must be in 2..65535");
  if (p.trials == 0) return COBEL_OK;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  COBEL_DISPATCH_A(p.world.n_actions, return launch<A>(p, st));
}
