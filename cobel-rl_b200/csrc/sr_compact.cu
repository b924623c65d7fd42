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

// ---------------------------------------------------------------------------
// Visited sets that do not fit on chip: sr_compact_large_kernel computes exactly what
// sr_compact_kernel<A, false> computes, with the per-agent tables (visited, rewards, model) left in
// HBM and one CTA per agent, so that the length-V row work of a step is spread over 256 threads.
// Every warp runs the agent's control flow redundantly (own draw window, same action), so all
// branches are CTA-uniform; shared memory holds only
//     slot[S]          global state -> local index (0xFFFF = not visited), rebuilt every launch
//     leaf_lo[L + 1]   first column of each leaf block of the pairwise tree over S columns
//     part[A][L]       leaf sums of one retrieve_q
// Q[a] is the pairwise sum of pairwise_sparse evaluated leaf-parallel: a leaf (<= 128 columns)
// scans its global states in order, takes the visited ones with rew != 0 and accumulates
// SRc[m_a][j] * rew[j] exactly as pairwise_sparse does; one lane per action then adds the leaf sums
// along the same tree.  Empty leaves and subtrees give 0.0 in both, and neither produces -0.0, so
// the result is bit-identical.
// ---------------------------------------------------------------------------
constexpr int kLargeThreads = 256;

// Leaf blocks of NumPy's pairwise tree over n_total elements, in order; writes their first indices to
// lo_out (if given) and returns their number.
__host__ __device__ inline int pairwise_leaves(int n_total, int* lo_out) {
  struct Frame { int lo, n; };
  Frame st[32];
  int sp = 0, L = 0;
  st[sp++] = Frame{0, n_total};
  while (sp > 0) {
    const Frame f = st[--sp];
    if (f.n <= 128) { if (lo_out) lo_out[L] = f.lo; ++L; continue; }
    int n2 = f.n / 2; n2 -= n2 % 8;
    st[sp++] = Frame{f.lo + n2, f.n - n2};          // right half is popped after the left one
    st[sp++] = Frame{f.lo, n2};
  }
  if (lo_out) lo_out[L] = n_total;
  return L;
}

// Adds leaf sums part[0..L) along the pairwise tree over n_total elements (the internal nodes of
// pairwise_sparse).
__device__ __noinline__ double pairwise_combine(const double* part, int n_total) {
  struct Frame { int n, phase; double left; };
  Frame st[32];
  int sp = 0, leaf = 0;
  double ret = 0.0;
  st[sp++] = Frame{n_total, 0, 0.0};
  while (sp > 0) {
    Frame& f = st[sp - 1];
    int n2 = f.n / 2; n2 -= n2 % 8;
    if (f.phase == 0) {
      if (f.n <= 128) { ret = part[leaf++]; --sp; continue; }
      f.phase = 1;
      st[sp++] = Frame{n2, 0, 0.0};
    } else if (f.phase == 1) {
      f.left = ret; f.phase = 2;
      st[sp++] = Frame{f.n - n2, 0, 0.0};
    } else {
      ret = xadd(f.left, ret); --sp;
    }
  }
  return ret;
}

struct LargeSmem {
  int slot, leaf_lo, part, q, bytes;
  LargeSmem(int S, int L, int A) {
    part = 0;                                        // [A][L] doubles
    q = part + A * L * 8;                            // [A] doubles
    leaf_lo = q + 8 * 8;                             // [L + 1] ints
    slot = leaf_lo + (L + 1) * 4;                    // [S] uint16
    bytes = slot + S * 2;
  }
};

template <int A>
__global__ void __launch_bounds__(kLargeThreads) sr_compact_large_kernel(const __grid_constant__ CobelSRCompactParams p,
                                                                         LargeSmem so, int L) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, K = p.world.n_starts, Vmax = p.max_visited;
  const int tid = threadIdx.x, lane = tid & 31;
  const int64_t n = blockIdx.x;
  double* part = reinterpret_cast<double*>(smem + so.part);
  double* qs = reinterpret_cast<double*>(smem + so.q);
  int32_t* leaf_lo = reinterpret_cast<int32_t*>(smem + so.leaf_lo);
  uint16_t* slot = reinterpret_cast<uint16_t*>(smem + so.slot);

  double* SRc = p.SRc + (size_t)n * Vmax * Vmax;
  double* rew = p.rewards + (size_t)n * Vmax;
  int32_t* vis = p.visited + (size_t)n * Vmax;
  int32_t* model = p.model + (size_t)n * Vmax * A;
  int V = p.n_visited[n];
  for (int g = tid; g < S; g += kLargeThreads) slot[g] = 0xFFFF;
  if (tid == 0) pairwise_leaves(S, leaf_lo);
  __syncthreads();
  for (int e = tid; e < V; e += kLargeThreads) slot[vis[e]] = (uint16_t)e;
  __syncthreads();

  DrawWindowT<true> win; win.init(p.stream, n, (uint64_t)p.stream.draw_count[n]);
  const double lr = p.lr[n], gamma = p.gamma[n];
  PolicyTab pt; pt.init(p.policy.kind, p.policy.param[n], lane);
  const bool learn = p.learn != 0;
  const CobelTrace& tr = p.trace;
  int64_t nsteps = 0;
  int flags = 0;

  // as in sr_compact_kernel; the new index, its identity row, zero column, self-loop model and zero
  // reward are written straight to HBM
  auto locate = [&](int g) -> int {
    const int e = slot[g];
    if (e != 0xFFFF) return e;
    if (V >= Vmax) { flags |= COBEL_FLAG_VISITED_OVERFLOW; return Vmax - 1; }
    const int v = V;
    for (int j = tid; j <= v; j += kLargeThreads) SRc[(size_t)v * Vmax + j] = j == v ? 1.0 : 0.0;
    for (int i = tid; i < v; i += kLargeThreads) SRc[(size_t)i * Vmax + v] = 0.0;
    if (tid == 0) { vis[v] = g; rew[v] = 0.0; }
    if (tid < A) model[(size_t)v * A + tid] = v;
    ++V;
    __syncthreads();                                 // every thread has read slot[g] before it changes
    if (tid == 0) slot[g] = (uint16_t)v;
    __syncthreads();
    return v;
  };

  for (int trial = 0; trial < p.trials; ++trial) {
    win.ensure(2, lane);
    int s = __ldg(p.world.starts + draw_integer(win.next(), K));
    int ls = locate(s);
    double treward = 0.0;
    int step = 0;
    for (;; ++step) {
      // ---- retrieve_q: leaf sums over the reward-carrying visited columns, then the tree -------------
      for (int it = tid; it < A * L; it += kLargeThreads) {
        const int a = it / L, l = it - a * L;
        const int lo = leaf_lo[l], hi = leaf_lo[l + 1], nl = hi - lo;
        const double* row = SRc + (size_t)model[(size_t)ls * A + a] * Vmax;
        double res = 0.0;
        if (nl < 8) {
          for (int g = lo; g < hi; ++g) {
            const int e = slot[g];
            if (e == 0xFFFF) continue;
            const double rv = rew[e];
            if (rv != 0.0) res = xadd(res, xmul(row[e], rv));
          }
        } else {
          double r[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
          const int main_end = hi - (nl & 7);
          for (int g0 = lo; g0 < main_end; g0 += 8) {
#pragma unroll
            for (int t = 0; t < 8; ++t) {
              const int e = slot[g0 + t];
              if (e == 0xFFFF) continue;
              const double rv = rew[e];
              if (rv != 0.0) r[t] = xadd(r[t], xmul(row[e], rv));
            }
          }
          res = xadd(xadd(xadd(r[0], r[1]), xadd(r[2], r[3])), xadd(xadd(r[4], r[5]), xadd(r[6], r[7])));
          for (int g = main_end; g < hi; ++g) {
            const int e = slot[g];
            if (e == 0xFFFF) continue;
            const double rv = rew[e];
            if (rv != 0.0) res = xadd(res, xmul(row[e], rv));
          }
        }
        part[it] = res;
      }
      __syncthreads();
      if (tid < A) qs[tid] = pairwise_combine(part + tid * L, S);
      __syncthreads();
      double row[A];
#pragma unroll
      for (int a = 0; a < A; ++a) row[a] = qs[a];
      // ---- action selection, environment step (every warp, same draws) ------------------------------
      win.ensure(2, lane);
      uint32_t mask = (1u << A) - 1u;
      if (p.action_mask) {
        mask = 0;
#pragma unroll
        for (int a = 0; a < A; ++a) mask |= (p.action_mask[(size_t)s * A + a] ? 1u : 0u) << a;
      }
      const int a = select_action_warp<A>(row, mask, pt, win.next(), lane);
      const int s2 = p.world.tp_off ? stochastic_successor(p.world, s * A + a, win.next()) : __ldg(p.world.succ + (size_t)s * A + a);
      const double r = __ldg(p.world.reward + s2);
      const int end = __ldg(p.world.terminal + s2);
      if (tr.step_sa && tid == 0) {
        if (nsteps < tr.step_cap) { tr.step_sa[n * tr.step_cap + nsteps] = s * A + a; if (tr.step_next) tr.step_next[n * tr.step_cap + nsteps] = s2; }
        else flags |= COBEL_FLAG_TRACE_OVERFLOW;
      }
      ++nsteps;
      int ls2 = ls;
      if (learn) {
        ls2 = locate(s2);
        // ---- SR.update on the visited columns: row ls from rows ls and ls2 ----------------------------
        const double* rs = SRc + (size_t)ls * Vmax;
        const double* rs2 = SRc + (size_t)ls2 * Vmax;
        double* wr = SRc + (size_t)ls * Vmax;
#pragma unroll 4
        for (int j = tid; j < V; j += kLargeThreads) {
          const double old = rs[j];
          const double x = end ? (j == ls2 ? 1.0 : 0.0) : rs2[j];
          double td = xadd(j == ls ? 1.0 : 0.0, xmul(gamma, x));
          td = xsub(td, old);
          wr[j] = xadd(old, xmul(lr, td));
        }
        if (tid == 0) {
          const double r0 = rew[ls2];
          rew[ls2] = xadd(r0, xmul(xsub(r, r0), lr));
          model[(size_t)ls * A + a] = ls2;
        }
        __syncthreads();
      } else if (!end && step + 1 != p.steps) {
        ls2 = locate(s2);
      }
      s = s2; ls = ls2;
      treward = xadd(treward, r);
      if (end || step + 1 == p.steps) break;
    }
    if (tid == 0) {
      tr.trial_steps[n * p.trials + trial] = step;
      tr.trial_reward[n * p.trials + trial] = treward;
    }
  }

  if (tid == 0) {
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
  if (sm > kMaxSmem) {
    const int L = pairwise_leaves(p.world.n_states, nullptr);
    const LargeSmem lo(p.world.n_states, L, A);
    COBEL_REQUIRE(lo.bytes <= kMaxSmem, COBEL_EUNSUPPORTED,
                  "max_visited %d needs the HBM-resident visited set, whose per-state slot map of %d states does not fit "
                  "in shared memory", p.max_visited, p.world.n_states);
    return launch_kernel(sr_compact_large_kernel<A>, (unsigned)p.n_agents, kLargeThreads, (size_t)lo.bytes, st, p, lo, L);
  }
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
