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
// pos[t] and val[t] are read through operator[] (arrays, or the accessors of sr_compact_op_kernel); each val[t] once.
template <class Pos, class Val>
__device__ __noinline__ double pairwise_sparse(Pos pos, Val val, int k, int n_total) {
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

// One agent's compact tables in HBM and its global -> local slot map in shared memory, as used by a CTA of
// kLargeThreads threads (sr_compact_large_kernel, sr_compact_op_kernel).
template <int A>
struct HbmAgent {
  double* SRc;
  double* rew;
  int32_t* vis;
  int32_t* model;
  uint16_t* slot;                                    // [S] local index of a global state, 0xFFFF = not visited
  int Vmax;

  __device__ HbmAgent(const CobelSRCompactParams& p, int64_t n, uint16_t* slot_)
      : SRc(p.SRc + (size_t)n * p.max_visited * p.max_visited), rew(p.rewards + (size_t)n * p.max_visited),
        vis(p.visited + (size_t)n * p.max_visited), model(p.model + (size_t)n * p.max_visited * A), slot(slot_),
        Vmax(p.max_visited) {}

  // rebuilds slot[] from the first V entries of visited[] (whole CTA)
  __device__ void build_slot(int S, int V) const {
    for (int g = threadIdx.x; g < S; g += kLargeThreads) slot[g] = 0xFFFF;
    __syncthreads();
    for (int e = threadIdx.x; e < V; e += kLargeThreads) slot[vis[e]] = (uint16_t)e;
    __syncthreads();
  }

  // as locate in sr_compact_kernel (whole CTA); the new index, its identity row, zero column, self-loop model and
  // zero reward are written straight to HBM
  __device__ int locate(int g, int& V, int& flags) const {
    const int tid = threadIdx.x;
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
  }
};

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

  const HbmAgent<A> ag(p, n, slot);
  double* SRc = ag.SRc;
  double* rew = ag.rew;
  int32_t* model = ag.model;
  int V = p.n_visited[n];
  if (tid == 0) pairwise_leaves(S, leaf_lo);
  ag.build_slot(S, V);

  DrawWindowT<true> win; win.init(p.stream, n, (uint64_t)p.stream.draw_count[n]);
  const double lr = p.lr[n], gamma = p.gamma[n];
  PolicyTab pt; pt.init(p.policy.kind, p.policy.param[n], lane);
  const bool learn = p.learn != 0;
  const CobelTrace& tr = p.trace;
  int64_t nsteps = 0;
  int flags = 0;
  auto locate = [&](int g) -> int { return ag.locate(g, V, flags); };

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

// ---------------------------------------------------------------------------
// Stand-alone SR.update / SR.retrieve_q on the compact tables (cobel_sr_compact_op).  The tables live in HBM for
// both fused kernels, so one kernel serves agents trained by either, at any max_visited.  One CTA of kLargeThreads
// per agent; shared memory holds the slot map (rebuilt from visited on every call) and, for RETRIEVE_Q, the local
// indices of the reward-carrying visited columns in global order:
//     wcount[kLargeThreads / 32] | slot[S] uint16 | cols[min(Vmax, S)] uint16
// ---------------------------------------------------------------------------
struct OpSmem {
  int slot, cols, bytes;
  OpSmem(int S, int n_cols) {
    slot = (kLargeThreads / 32) * 4;
    cols = slot + S * 2;
    bytes = cols + n_cols * 2;
  }
};

// pairwise_sparse's operands over cols[]: the global state of column t, and SR[m][j] * rew[j] formed when it is read
struct ColPos {
  const uint16_t* cols;
  const int32_t* vis;
  __device__ int operator[](int t) const { return __ldg(vis + cols[t]); }
};
struct ColProd {
  const uint16_t* cols;
  const double* row;
  const double* rew;
  __device__ double operator[](int t) const { const int e = cols[t]; return xmul(row[e], __ldg(rew + e)); }
};

template <int A>
__global__ void __launch_bounds__(kLargeThreads) sr_compact_op_kernel(const __grid_constant__ CobelSRCompactParams p,
                                                                      OpSmem so, int op, CobelExperiences e,
                                                                      const int32_t* states, int n_query, double* q_out) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, Vmax = p.max_visited;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t n = blockIdx.x;
  int32_t* wcount = reinterpret_cast<int32_t*>(smem);
  uint16_t* slot = reinterpret_cast<uint16_t*>(smem + so.slot);
  uint16_t* cols = reinterpret_cast<uint16_t*>(smem + so.cols);
  const HbmAgent<A> ag(p, n, slot);
  int V = p.n_visited[n];
  ag.build_slot(S, V);

  if (op == COBEL_OP_STORE) {
    // ---- SR.update (agent/sr.py:255-286) as one learning step of the fused kernels: s, then s', are located or
    // inserted; row ls from rows ls and ls'; then rew[ls'] and model[ls][a] ----------------------------------------
    const int64_t i = n * e.batch;
    const int s = e.state[i], a = e.action[i], s2 = e.next_state[i];
    const bool nonterminal = e.terminal[i] != 0;
    const double r = e.reward[i], lr = p.lr[n], gamma = p.gamma[n];
    int flags = 0;
    const int ls = ag.locate(s, V, flags);
    const int ls2 = ag.locate(s2, V, flags);
    const double* rs = ag.SRc + (size_t)ls * Vmax;
    const double* rs2 = ag.SRc + (size_t)ls2 * Vmax;
    double* wr = ag.SRc + (size_t)ls * Vmax;
    for (int j = tid; j < V; j += kLargeThreads) {
      const double old = rs[j];
      const double x = nonterminal ? rs2[j] : (j == ls2 ? 1.0 : 0.0);
      double td = xadd(j == ls ? 1.0 : 0.0, xmul(gamma, x));
      td = xsub(td, old);
      wr[j] = xadd(old, xmul(lr, td));
    }
    if (tid == 0) {
      const double r0 = ag.rew[ls2];
      ag.rew[ls2] = xadd(r0, xmul(xsub(r, r0), lr));
      ag.model[(size_t)ls * A + a] = ls2;
      p.n_visited[n] = V;
      if (p.trace.flags && flags) p.trace.flags[n] |= flags;
    }
    return;
  }

  // ---- SR.retrieve_q (agent/sr.py:288-308) for n_query states: one ordered pass over slot[] lists the visited
  // columns with rew != 0 in global order (block-wide stream compaction, one tile of kLargeThreads states at a time) --
  int k = 0;
  for (int g0 = 0; g0 < S; g0 += kLargeThreads) {
    const int g = g0 + tid;
    const int ev = g < S ? slot[g] : 0xFFFF;
    const bool nz = ev != 0xFFFF && ag.rew[ev] != 0.0;
    const unsigned b = __ballot_sync(kFull, nz);
    if (lane == 0) wcount[warp] = __popc(b);
    __syncthreads();
    int off = k;
#pragma unroll
    for (int w = 0; w < kLargeThreads / 32; ++w) {
      const int c = wcount[w];
      off += w < warp ? c : 0;
      k += c;
    }
    if (nz) cols[off + __popc(b & ((1u << lane) - 1u))] = (uint16_t)ev;
    __syncthreads();                                 // wcount is rewritten by the next tile
  }
  // Q[b][a] = pairwise_sparse over those columns of row m(s_b, a).  An unvisited s_b has the row e_{s_b} and zero
  // reward: every product is a signed zero and the sum is +0.0, exactly what pairwise_sparse returns for them.
  const ColPos pos{cols, ag.vis};
  const int64_t items = (int64_t)n_query * A;
  for (int64_t it = tid; it < items; it += kLargeThreads) {
    const int64_t b = it / A;
    const int a = (int)(it - b * A);
    const int ls = slot[states[n * n_query + b]];
    double q = 0.0;
    if (ls != 0xFFFF) {
      const ColProd val{cols, ag.SRc + (size_t)ag.model[(size_t)ls * A + a] * Vmax, ag.rew};
      q = pairwise_sparse(pos, val, k, S);
    }
    q_out[n * items + it] = q;
  }
}

template <int A>
int launch_op(const CobelSRCompactParams& p, int op, const CobelExperiences& e, const int32_t* states, int n_query,
              double* q_out, cudaStream_t st) {
  const int S = p.world.n_states;
  const int n_cols = op == COBEL_OP_RETRIEVE_Q ? (p.max_visited < S ? p.max_visited : S) : 0;
  const OpSmem so(S, n_cols);
  if (op == COBEL_OP_STORE)
    COBEL_REQUIRE(so.bytes <= kMaxSmem, COBEL_EUNSUPPORTED,
                  "cobel_sr_compact_op(STORE): the slot map of %d states needs %d bytes of shared memory (at most %d)",
                  S, so.bytes, kMaxSmem);
  else
    COBEL_REQUIRE(so.bytes <= kMaxSmem, COBEL_EUNSUPPORTED,
                  "cobel_sr_compact_op(RETRIEVE_Q): the slot map of %d states and the list of up to %d reward-carrying "
                  "states need %d bytes of shared memory (at most %d)", S, n_cols, so.bytes, kMaxSmem);
  return launch_kernel(sr_compact_op_kernel<A>, (unsigned)p.n_agents, kLargeThreads, (size_t)so.bytes, st, p, so, op,
                       e, states, n_query, q_out);
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

extern "C" int cobel_sr_compact_op(const CobelSRCompactParams* pp, int op, const CobelExperiences* e,
                                   const int32_t* states, int32_t n_query, double* q_out, void* stream) {
  COBEL_REQUIRE(pp != nullptr, COBEL_EINVAL, "null params");
  const CobelSRCompactParams& p = *pp;
  COBEL_REQUIRE(p.n_agents > 0 && p.world.n_states > 0, COBEL_EINVAL, "null / empty params");
  COBEL_REQUIRE(p.SRc && p.rewards && p.model && p.visited && p.n_visited && p.lr && p.gamma, COBEL_EINVAL,
                "agent tables missing");
  COBEL_REQUIRE(p.max_visited >= 2 && p.max_visited <= 65535, COBEL_EINVAL, "max_visited must be in 2..65535");
  const bool store_ok = op == COBEL_OP_STORE && e && e->batch > 0 && e->state && e->action && e->reward &&
                        e->next_state && e->terminal;
  COBEL_REQUIRE(store_ok || (op == COBEL_OP_RETRIEVE_Q && states && q_out && n_query > 0), COBEL_EINVAL,
                "cobel_sr_compact_op: op must be COBEL_OP_STORE (SR.update, with an experience) or COBEL_OP_RETRIEVE_Q "
                "(with states, n_query > 0 and q_out)");
  const CobelExperiences none{};
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  COBEL_DISPATCH_A(p.world.n_actions, return launch_op<A>(p, op, e ? *e : none, states, n_query, q_out, st));
}
