// sfma.cu -- K5: SFMA.train()/test() (Dyna-Q with SFMA replay: strength x similarity x
// inhibition sampling over a state-similarity metric D) for N independent agents in one launch.
//
// Reference: agent/sfma.py:233-458 (trial loop, replay, masked update_q) and
// memory/sfma.py:195-373 (store, replay, softmax).  Semantics: SURVEY.md Appendix A.6.
//
// Mapping: one CTA per agent; all per-agent tables (Q, M.rewards, M.states|terminals, C, I and
// the priority scratch R) live in shared memory, the shared similarity matrix D[S,S] is read
// from HBM/L2 one row at a time (coalesced).  The online steps of a trial are executed by
// warp 0 (warp-uniform, as in the Dyna-Q kernel); each replay reactivation is a CTA-wide pass
// over the S*A experiences: priority R = C*D*(1-I) -> threshold -> max -> exp -> inverse-CDF
// draw by a block scan -> inhibition update.  The replayed TD updates are applied afterwards,
// in order, by the level-parallel batch of warp_agent.cuh.
//
// Exactness: every quantity that reaches Q, C, I or an integer is computed with the
// reference's operation order; exp() and the CDF prefix sums are not bit-identical to NumPy's
// and only decide the sampled index, so a draw that falls within 1e-12 of a bin edge raises
// COBEL_FLAG_CDF_NEAR_TIE instead of silently risking a different index.
#include "warp_agent.cuh"
#include "thread_agent.cuh"

namespace {

enum { MODE_DEFAULT = 0, MODE_FORWARD, MODE_REVERSE, MODE_BLEND_FORWARD, MODE_BLEND_REVERSE, MODE_INTERPOLATE, MODE_SWEEPING };

struct SfmaSmem {
  int q, mr, c, t, r, inh, part, mx, mbits, rep, lst, cdf, bytes;
  __host__ __device__ SfmaSmem(int S, int A, int T, int B, bool recency, bool random_replay) {
    const int N = S * A;
    q = 0;
    mr = q + N * 8;
    c = mr + N * 8;
    t = c + N * 8;
    r = t + (recency ? N * 8 : 0);
    inh = r + N * 8;
    part = inh + S * 8;
    rep = part + (T + 32) * 8;
    mx = rep + ((B + 1) & ~1) * 4;
    mbits = mx + N * 2;
    lst = (mbits + S + 3) & ~3;
    cdf = (lst + N * 4 + 7) & ~7;
    bytes = (cdf + (random_replay ? N * 8 : 0) + 15) & ~15;
  }
};

struct BlockShared {
  double u, total, target;
  int idx, flag, action, last, brk;
};

// Exclusive block scan of one double per thread (T <= 1024); also returns the grand total.
COBEL_DEV double block_exclusive_scan(double v, double* part, int tid, int T, double& total) {
  const int lane = tid & 31, warp = tid >> 5, nw = T >> 5;
  double inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const double o = shfl_f64_up(inc, d);
    if (lane >= d) inc += o;
  }
  if (lane == 31) part[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    double w = lane < nw ? part[lane] : 0.0;
    double winc = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const double o = shfl_f64_up(winc, d);
      if (lane >= d) winc += o;
    }
    if (lane < nw) part[lane] = winc - w;          // exclusive offset of each warp
    if (lane == 31) part[32] = winc;               // grand total
  }
  __syncthreads();
  total = part[32];
  const double res = part[warp] + (inc - v);
  __syncthreads();                                  // part[] may be reused by the caller
  return res;
}

// integer exclusive block scan (T <= 1024)
COBEL_DEV int block_exclusive_scan_int(int v, double* part, int tid, int T, int& total) {
  int* ip = reinterpret_cast<int*>(part);
  const int lane = tid & 31, warp = tid >> 5, nw = T >> 5;
  int inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int o = __shfl_up_sync(kFull, inc, d);
    if (lane >= d) inc += o;
  }
  if (lane == 31) ip[warp] = inc;
  __syncthreads();
  int off = 0, tot = 0;
  for (int w = 0; w < nw; ++w) { if (w < warp) off += ip[w]; tot += ip[w]; }
  total = tot;
  __syncthreads();
  return off + inc - v;
}

// Inverse-CDF draw over non-negative weights w[0..N): the first i whose running sum / total
// exceeds u  (NumPy: searchsorted(cumsum(p)/cumsum(p)[-1], u, 'right') with p = w/sum(w)).
COBEL_DEV int block_sample(const double* w, int N, double u, double* part, BlockShared* sh, int tid, int T, int& flags) {
  const int chunk = (N + T - 1) / T;
  const int lo = tid * chunk < N ? tid * chunk : N, hi = lo + chunk < N ? lo + chunk : N;
  double local = 0.0;
#pragma unroll 1
  for (int i = lo; i < hi; ++i) local += w[i];
  double total;
  const double excl = block_exclusive_scan(local, part, tid, T, total);
  const double target = u * total;
  const double tol = 1e-12 * total;
  if (tid == 0) { sh->idx = 0x7fffffff; sh->flag = 0; }
  __syncthreads();
  // owner = the first thread whose running sum passes the target
  if (local > 0.0 && excl + local > target) atomicMin(&sh->idx, tid);
  __syncthreads();
  const int owner = sh->idx;
  __syncthreads();
  if (owner == 0x7fffffff) {                       // u*total rounded up to the total: the last positive weight
    if (tid == 0) {
      int f = N - 1;
      while (f > 0 && !(w[f] > 0.0)) --f;
      sh->idx = f; sh->flag = 1;
    }
  } else if (tid == owner) {
    double acc = excl;
    int found = -1, lastpos = lo;
    bool near = fabs(excl - target) < tol;
#pragma unroll 1
    for (int i = lo; i < hi; ++i) {
      if (!(w[i] > 0.0)) continue;
      lastpos = i;
      acc += w[i];
      if (fabs(acc - target) < tol) near = true;
      if (found < 0 && acc > target) found = i;
    }
    sh->idx = found >= 0 ? found : lastpos;
    if (near || found < 0) sh->flag = 1;
  }
  __syncthreads();
  const int idx = sh->idx;
  if (sh->flag) flags |= COBEL_FLAG_CDF_NEAR_TIE;
  __syncthreads();
  return idx;
}

// ---------------------------------------------------------------------------
// Split path (the common configuration: no per-step decay of C or T, no strength modulation that touches every
// experience).  A trial is two launches:
//   sfma_step_kernel    ONE THREAD PER AGENT: reset + the online steps.  A step reads one Q row, draws an action,
//                       looks the successor up and updates one entry each of Q, M.rewards, M.states, M.terminals and
//                       C -- a dozen scattered 8-byte accesses to the agent's tables in HBM and ~150 scalar
//                       instructions.  In the fused kernel warp 0 of the agent's CTA does this while 7 warps wait at
//                       a barrier (61 % of the kernel's time at 3 CTAs per SM, profiles/r1_sfma_v2.txt); here a warp
//                       advances 32 agents at once and every agent of the batch is in flight.
//   sfma_replay_kernel  ONE CTA PER AGENT: SFMAMemory.replay + the replayed Q updates.  Only what a replay reads is
//                       staged: the compact list of experienced (s, a) with their strengths and next states, the
//                       inhibition vector and the priority scratch (41 KB at 20x20 instead of 67 KB: 5 CTAs per SM);
//                       Q stays in HBM and receives the <= batch updates at the end.
// The per-agent state between the launches (current / last state, counters) travels in CobelSFMAParams.carry.
// ---------------------------------------------------------------------------
struct SfmaPhase {
  int init;           // step kernel: first launch of a call (the carry's counters restart)
  int reset;          // step kernel: draw the start state of the first trial of this launch
  int n_trials;       // step kernel: trials run by this launch (0: reset only; several only without any replay)
  int trial;          // index of the (first) trial (trace rows)
  int start_replay;   // replay kernel: the trace-only replay at trial start (cur = start state, no Q updates)
  int list_cap;       // replay kernel: capacity of the list of experienced (s, a) (ReplaySmem)
};

template <int A>
__global__ void __launch_bounds__(64) sfma_step_kernel(const __grid_constant__ CobelSFMAParams p, const __grid_constant__ SfmaPhase ph) {
  const int64_t n = (int64_t)blockIdx.x * 64 + threadIdx.x;
  if (n >= p.n_agents) return;
  const int S = p.world.n_states, K = p.world.n_starts, N = S * A;
  const size_t g0 = (size_t)n * N;
  double* Q = p.Q + g0;
  double* Mr = p.Mr + g0;
  int32_t* Ms = p.Ms + g0;
  int32_t* Mt = p.Mt + g0;
  double* C = p.C + g0;
  const uint8_t* amask = p.action_mask ? p.action_mask + n * p.mask_agent_stride : nullptr;
  int64_t* carry = p.carry + n * 4;        // [0] current state / last state (-1: timed out)  [1] steps  [2] replayed  [3] replay calls
  const CobelTrace& tr = p.trace;
  Rng rng; rng.init(p.stream, n);
  const bool learn = p.learn != 0;
  const int kind = p.policy.kind;
  const double par = p.policy.param[n];
  const double lr = p.lr[n], gamma = p.gamma[n], mlr = p.mem_lr[n];
  const int mf = p.mod_flags;
  int flags = 0;
  if (ph.init) { carry[0] = 0; carry[1] = 0; carry[2] = 0; carry[3] = 0; }
  int s = (int)carry[0];
  for (int t = 0; t < ph.n_trials || t == 0; ++t) {
    if (ph.reset || t > 0) s = __ldg(p.world.starts + draw_integer(rng.next(), K));
    if (t >= ph.n_trials) break;
    int64_t nsteps = carry[1];
    double tdacc = p.td_acc ? p.td_acc[n] : 0.0;
    double treward = 0.0;
    int step = 0, last = -1;
    // The tables live in HBM and a step touches a handful of their entries, so what a step costs is its DEPENDENT
    // DRAM round trips: all loads of a step that do not depend on one another (M.rewards[s,a], C[a,s], Q[s',:]) are
    // issued together as soon as the action is known, before any store, and the row Q[s',:] is carried over as the
    // next step's Q[s,:] -- one round trip per step instead of four.
    double row[A];
    load_row_t<A>(Q + (size_t)s * A, row);
    for (;; ++step) {
      const int a = select_action_thread<A>(row, mask_bits<A>(amask, s), kind, par, rng.next());
      const int s2 = p.world.tp_off ? stochastic_successor_t(p.world, s * A + a, rng.next()) : __ldg(p.world.succ + s * A + a);
      const double r = __ldg(p.world.reward + s2);
      const int end = __ldg(p.world.terminal + s2);
      const int nt = 1 - end;
      if (tr.step_sa) {
        if (nsteps < tr.step_cap) { tr.step_sa[n * tr.step_cap + nsteps] = s * A + a; if (tr.step_next) tr.step_next[n * tr.step_cap + nsteps] = s2; }
        else flags |= COBEL_FLAG_TRACE_OVERFLOW;
      }
      ++nsteps;
      double row2[A];
      if (learn) {
        // SFMAMemory.store (memory/sfma.py:206-215; decay_strength == 1 and M.T is not tracked on this path), then
        // SFMA.update_q (agent/sfma.py:423-458): max over the unmasked actions of s'
        const double m0 = Mr[s * A + a];                           // ---- loads ----
        double cs[A];
        if (mf & COBEL_SFMA_MOD_STATE) {
#pragma unroll
          for (int x = 0; x < A; ++x) cs[x] = C[x * S + s];
        } else {
          cs[0] = C[a * S + s];
        }
        load_row_t<A>(Q + (size_t)s2 * A, row2);
        const uint32_t mb2 = mask_bits<A>(amask, s2);
        Mr[s * A + a] = xadd(m0, xmul(mlr, xsub(r, m0)));          // ---- stores ----
        Ms[s * A + a] = s2;
        Mt[s * A + a] = nt;
        if (mf & COBEL_SFMA_MOD_STATE) {                           // memory/sfma.py:233-236: every action of s, after the store
#pragma unroll
          for (int x = 0; x < A; ++x) {
            double c = cs[x];
            if (x == a) {
              c = xadd(c, p.c_step);
              if (mf & COBEL_SFMA_MOD_REWARD_LOCAL) c = xadd(c, xmul(r, p.reward_modulation));
            }
            C[x * S + s] = xadd(c, 1.0);
          }
        } else {
          double c = xadd(cs[0], p.c_step);
          if (mf & COBEL_SFMA_MOD_REWARD_LOCAL) c = xadd(c, xmul(r, p.reward_modulation));   // memory/sfma.py:216-218
          C[a * S + s] = c;
        }
        // td = r + (gamma * terminal) * max_{valid} Q[s'] - Q[s,a]; Q[s,a] += lr * td  (Q[s,:] is `row`)
        double mx = -__longlong_as_double(0x7FF0000000000000ll);
#pragma unroll
        for (int x = 0; x < A; ++x) mx = (mb2 >> x & 1u) ? xmax(mx, row2[x]) : mx;
        const double q = pick_reg<A>(row, a);
        double td = xadd(r, xmul(nt ? gamma : 0.0, mx));
        td = xsub(td, q);
        const double qn = xadd(q, xmul(lr, td));
        Q[(size_t)s * A + a] = qn;
        if (s2 == s) {                                             // the carried row must see the update
#pragma unroll
          for (int x = 0; x < A; ++x) row2[x] = x == a ? qn : row2[x];
        }
        tdacc = xadd(tdacc, fabs(td));
      } else {
        load_row_t<A>(Q + (size_t)s2 * A, row2);
      }
#pragma unroll
      for (int x = 0; x < A; ++x) row[x] = row2[x];
      s = s2;
      treward = xadd(treward, r);
      if (end) last = s2;
      if (end || step + 1 == p.steps) break;
    }
    tr.trial_steps[n * p.trials + ph.trial + t] = step;
    tr.trial_reward[n * p.trials + ph.trial + t] = treward;
    tr.n_steps[n] += nsteps - carry[1];
    carry[1] = nsteps;
    if (p.td_acc) p.td_acc[n] = tdacc;
    s = last;
  }
  carry[0] = s;
  p.stream.draw_count[n] = (int64_t)rng.k;
  if (flags && tr.flags) tr.flags[n] |= flags;
}

struct ReplaySmem {
  int l, cc, msc, r, inh, part, rep, mbits, cdf, bytes, cap;
  // cap = capacity of the list of experienced (s, a): all S*A of them when that fits, else what shared memory
  // holds (an agent that has experienced more raises COBEL_FLAG_REPLAY_OVERFLOW)
  __host__ __device__ ReplaySmem(int S, int A, int T, int B, bool random_replay, int cap_ = -1) {
    const int N = S * A;
    cap = cap_ < 0 ? N : cap_;
    const int R = cap > S ? cap : S;         // the priority scratch also hosts the 2 S dependency-mask words (8 S bytes)
    r = 0;                                   // priority scratch [nnz] (aliased by the dependency masks of the TD batch)
    cc = r + R * 8;                          // strengths of the listed experiences
    inh = cc + cap * 8;                      // I [S]
    part = inh + S * 8;                      // scan partials
    cdf = part + (T + 32) * 8;               // random replay: m-fold sums of fl(1 / n_valid)
    l = cdf + (random_replay ? N * 8 : 0);   // experienced experiences: action << 16 | state, ascending flat index
    rep = l + cap * 4;                       // reactivated flat indices of one replay
    msc = rep + ((B + 1) & ~1) * 4;          // next state of the listed experiences
    mbits = msc + ((cap + 1) & ~1) * 2;      // valid-action bits per state
    bytes = (mbits + S + 15) & ~15;
  }
  // the largest list capacity whose layout fits into `limit` bytes
  static int fit(int S, int A, int T, int B, bool random_replay, int limit) {
    const int N = S * A;
    if (ReplaySmem(S, A, T, B, random_replay).bytes <= limit) return N;
    int lo = 0, hi = N;
    while (lo < hi) {
      const int mid = (lo + hi + 1) / 2;
      if (ReplaySmem(S, A, T, B, random_replay, mid).bytes <= limit) lo = mid; else hi = mid - 1;
    }
    return lo;
  }
};

#ifndef SFMA_REPLAY_MINB
#define SFMA_REPLAY_MINB 4
#endif
template <int A>
__global__ void __launch_bounds__(256, SFMA_REPLAY_MINB) sfma_replay_kernel(const __grid_constant__ CobelSFMAParams p, const __grid_constant__ SfmaPhase ph) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ BlockShared sh;
  const int S = p.world.n_states, N = S * A, B = p.batch;
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int64_t n = blockIdx.x;
  const ReplaySmem so(S, A, T, B, p.random_replay != 0, ph.list_cap);
  double* R = reinterpret_cast<double*>(smem + so.r);
  double* Cc = reinterpret_cast<double*>(smem + so.cc);
  double* I = reinterpret_cast<double*>(smem + so.inh);
  double* part = reinterpret_cast<double*>(smem + so.part);
  double* cdft = reinterpret_cast<double*>(smem + so.cdf);
  uint32_t* L = reinterpret_cast<uint32_t*>(smem + so.l);
  int32_t* rep = reinterpret_cast<int32_t*>(smem + so.rep);
  uint16_t* Msc = reinterpret_cast<uint16_t*>(smem + so.msc);
  uint8_t* mbits = smem + so.mbits;
  uint32_t* wm = reinterpret_cast<uint32_t*>(R);
  uint32_t* rm = wm + S;

  const size_t g0 = (size_t)n * N;
  double* Q = p.Q + g0;
  const double* Mr = p.Mr + g0;
  const int32_t* Ms = p.Ms + g0;
  const int32_t* Mt = p.Mt + g0;
  const double* Cg = p.C + g0;
  const uint8_t* amask = p.action_mask ? p.action_mask + n * p.mask_agent_stride : nullptr;
  int64_t* carry = p.carry + n * 4;
  const CobelTrace& tr = p.trace;
  const bool masked = amask != nullptr;
  const bool apply_updates = ph.start_replay == 0;
  // agent.random batches (retrieve_random_batch); start_replay == 2: the stand-alone memory call, without Q updates
  const bool random_path = p.random_replay && (apply_updates || ph.start_replay == 2);
  const double lr = apply_updates ? p.lr[n] : 0.0, gamma = apply_updates ? p.gamma[n] : 0.0;
  const double beta = p.beta, thr = p.threshold, dinh = p.decay_inhibition;
  const double* D = p.D;
  const int mf = p.mod_flags;
  double cmax = 1.0, dmax = 1.0;
  int mode = p.mode;
  int64_t nrep = carry[2], ncalls = carry[3];
  const int64_t nrep0 = nrep;
  const int last = (int)carry[0];
  int flags = 0;
  DrawWindow win; win.init(p.stream, n, (uint64_t)p.stream.draw_count[n]);      // used by warp 0 only
  double tdacc = p.td_acc ? p.td_acc[n] : 0.0;                                   // agent.td (maintained by warp 0)

#pragma unroll 1
  for (int e = tid; e < S; e += T) mbits[e] = (uint8_t)mask_bits<A>(amask, e);
  __syncthreads();

  auto acc_td = [&](double tdl, bool active) {
    if (!p.td_acc) return;
    const unsigned act = __ballot_sync(kFull, active);
#pragma unroll 1
    for (int l = 0; l < 32 && (act >> l & 1u); ++l) tdacc = xadd(tdacc, fabs(shfl_f64(tdl, l)));
  };
  // the replayed TD updates, in order, on the Q table in HBM (agent/sfma.py:416-419); warp 0
  auto apply_batch = [&](int count) {
#pragma unroll 1
    for (int e = tid; e < 2 * S; e += T) wm[e] = 0;                        // wm, rm alias R
    __syncthreads();
    if (warp == 0 && apply_updates) {
#pragma unroll 1
      for (int b0 = 0; b0 < count; b0 += 32) {
        const bool active = b0 + lane < count;
        int es = 0, ea = 0, es2 = 0, ent = 0;
        double er = 0.0;
        if (active) {
          const int e = rep[b0 + lane];
          ea = e / S; es = e - ea * S;
          er = Mr[es * A + ea];
          es2 = Ms[es * A + ea]; ent = Mt[es * A + ea] ? 1 : 0;
        }
        double tdl = 0.0;
        td_batch_level_parallel<A>(Q, wm, rm, S, lane, active, es, ea, er, es2, ent, lr, gamma,
                                   masked ? mbits : nullptr, &tdl);
        acc_td(tdl, active);
      }
    }
  };
  auto log_replay = [&](int count) {
    if (tr.replay_idx)
#pragma unroll 1
      for (int j = tid; j < count; j += T) {
        if (nrep + j < tr.replay_cap) tr.replay_idx[n * tr.replay_cap + nrep + j] = rep[j];
        else flags |= COBEL_FLAG_TRACE_OVERFLOW;
      }
    if (tr.replay_len && tid == 0) {
      if (ncalls < tr.replay_calls_cap) tr.replay_len[n * tr.replay_calls_cap + ncalls] = count;
      else flags |= COBEL_FLAG_TRACE_OVERFLOW;
    }
    nrep += count;
    ++ncalls;
  };

  if (!ph.start_replay && p.dynamic) {
    // agent/sfma.py:311-318: p('reverse') = 1 / (1 + exp(-(5 td - 2))), one categorical draw over
    // [p, 1 - p] (cdf normalised by its last entry), the accumulator restarts
    if (warp == 0) {
      win.ensure(1, lane);
      const double u = win.next();
      const double pm = xdiv(1.0, xadd(1.0, exp(-xsub(xmul(tdacc, 5.0), 2.0))));
      const double c0 = xdiv(pm, xadd(pm, xsub(1.0, pm)));
      if (fabs(c0 - u) < 1e-12) flags |= COBEL_FLAG_CDF_NEAR_TIE;      // exp() is not NumPy's bit for bit
      tdacc = 0.0;
      if (lane == 0) sh.idx = c0 > u ? MODE_REVERSE : MODE_DEFAULT;
    }
    __syncthreads();
    mode = sh.idx;
    if (p.trial_mode && tid == 0) p.trial_mode[n * p.trials + ph.trial] = mode;
    __syncthreads();
  }

  // similarity of experience (a, s') with modelled next state ms to the current experience, by replay mode
  // (memory/sfma.py:283-306)
  auto dvec = [&](int sp, int ms, int cur, int nxt) -> double {
    const double* Dc = D + (size_t)cur * S;
    const double* Dn = D + (size_t)nxt * S;
    auto dc = [&](int x) -> double { return (mf & COBEL_SFMA_D_NORMALIZE) ? xdiv(Dc[x], dmax) : Dc[x]; };
    switch (mode) {
      case MODE_FORWARD: return Dn[sp];
      case MODE_REVERSE: return dc(ms);
      case MODE_BLEND_FORWARD: return xadd(dc(sp), xmul(p.blend, Dn[sp]));
      case MODE_BLEND_REVERSE: return xadd(dc(sp), xmul(p.blend, dc(ms)));
      case MODE_INTERPOLATE: return xadd(xmul(p.interp_fwd, Dn[sp]), xmul(p.interp_rev, dc(ms)));
      case MODE_SWEEPING: return Dn[ms];
      default: return dc(sp);
    }
  };

  const int n_replays = ph.start_replay ? 1 : p.nb_replays;
  for (int rpl = 0; rpl < n_replays; ++rpl) {
    if (random_path) {
      // agent.random: uniform batches over the unmasked experiences (retrieve_random_batch, memory/sfma.py:375-416):
      // probs = mask / sum(mask); NumPy's choice() searches u in the m-fold sequential sums of fl(1 / n_valid)
      if (tid == 0) {
        int m = 0;
        for (int a = 0; a < A; ++a)
          for (int sp = 0; sp < S; ++sp)
            if (mbits[sp] >> a & 1) ++m;
        const double pv = xdiv(1.0, int_to_f64(m));
        double c = 0.0;
        for (int j = 0; j < m; ++j) { c = xadd(c, pv); cdft[j] = c; }
        sh.idx = m;
      }
      __syncthreads();
      const int nvalid = sh.idx;
      __syncthreads();
      if (warp == 0) {
        const double tot = cdft[nvalid - 1];
#pragma unroll 1
        for (int b0 = 0; b0 < B; b0 += 32) {
          const int nb = B - b0 < 32 ? B - b0 : 32;
          win.ensure(nb, lane);
          const double u = win.peek(lane < nb ? lane : 0);
          win.advance(nb);
          if (lane < nb) {
            int lo = 0, hi = nvalid - 1;                       // invariant: answer in [lo, hi]
            while (lo < hi) {
              const int mid = (lo + hi) >> 1;
              if (xdiv(cdft[mid], tot) > u) hi = mid; else lo = mid + 1;
            }
            int m = lo, e = -1;                                // m-th valid experience in F order
            for (int a = 0; a < A && e < 0; ++a)
              for (int sp = 0; sp < S; ++sp)
                if ((mbits[sp] >> a & 1) && m-- == 0) { e = a * S + sp; break; }
            rep[b0 + lane] = e;
          }
        }
      }
      __syncthreads();
      log_replay(B);
      apply_batch(B);
      __syncthreads();
      continue;
    }
    if (warp == 0) {
      win.ensure(2, lane);
      const int act0 = draw_integer(win.next(), A);                        // sfma.py:264 (always drawn)
      double u = 0.0;
      if (last < 0) u = win.next();                                        // sfma.py:272
      if (lane == 0) { sh.action = act0; sh.u = u; }
    }
    __syncthreads();
    int cur = last, action = sh.action;
    // Experiences that were never stored have strength 0, hence priority 0 and weight exp(0) - 1 = 0:
    // they can never be drawn and add exact zeros to every sum.  All passes below run over the compact,
    // index-ordered list L of experiences with C > 0 (C is constant during a replay).
    int nnz;
    {
      const int chunk = (N + T - 1) / T;
      const int lo = tid * chunk < N ? tid * chunk : N;
      int hi = lo + chunk < N ? lo + chunk : N;
      int cnt = 0;
#pragma unroll 1
      for (int i = lo; i < hi; ++i) cnt += Cg[i] > 0.0 ? 1 : 0;
      int off = block_exclusive_scan_int(cnt, part, tid, T, nnz);
      if (nnz > so.cap) {                                                  // more experienced (s, a) than the list holds
        flags |= COBEL_FLAG_REPLAY_OVERFLOW;
        nnz = 0; hi = lo;
      }
#pragma unroll 1
      for (int i = lo; i < hi; ++i) {
        const double c = Cg[i];
        if (c > 0.0) {
          const int a = i / S, sp = i - a * S;
          L[off] = ((uint32_t)a << 16) | (uint32_t)sp;
          Cc[off] = c;
          Msc[off] = (uint16_t)Ms[sp * A + a];
          ++off;
        }
      }
    }
    __syncthreads();
    if (mf & COBEL_SFMA_C_NORMALIZE) {                                     // np.amax(C): C is constant during a replay
      double lm = -__longlong_as_double(0x7FF0000000000000ll);
#pragma unroll 1
      for (int e = tid; e < N; e += T) lm = Cg[e] > lm ? Cg[e] : lm;
      for (int d = 16; d > 0; d >>= 1) { const double o = shfl_f64_xor(lm, d); lm = o > lm ? o : lm; }
      if (lane == 0) part[warp] = lm;
      __syncthreads();
      cmax = part[0];
      for (int w = 1; w < (T >> 5); ++w) cmax = part[w] > cmax ? part[w] : cmax;
      __syncthreads();
    }
    if (cur < 0) {                                                         // start ~ clip(C, 0) / sum
#pragma unroll 1
      for (int j = tid; j < nnz; j += T) R[j] = Cc[j];
      __syncthreads();
      const uint32_t l = L[block_sample(R, nnz, sh.u, part, &sh, tid, T, flags)];
      cur = l & 0xFFFF; action = l >> 16;
    }
    int nxt = Ms[cur * A + action];
#pragma unroll 1
    for (int e = tid; e < S; e += T) I[e] = 0.0;                           // sfma.py:277
    __syncthreads();
    int count = 0;
    const int nw = T >> 5, chunk = (nnz + T - 1) / T;
    const int clo = tid * chunk < nnz ? tid * chunk : nnz, chi = clo + chunk < nnz ? clo + chunk : nnz;
    for (int it = 0; it < B; ++it) {
      if (mf & COBEL_SFMA_D_NORMALIZE) {                                   // np.amax(D[current_state])
        const double* Dc = D + (size_t)cur * S;
        double lm = -__longlong_as_double(0x7FF0000000000000ll);
#pragma unroll 1
        for (int e = tid; e < S; e += T) lm = Dc[e] > lm ? Dc[e] : lm;
        for (int d = 16; d > 0; d >>= 1) { const double o = shfl_f64_xor(lm, d); lm = o > lm ? o : lm; }
        if (lane == 0) part[warp] = lm;
        __syncthreads();
        dmax = part[0];
        for (int w = 1; w < (T >> 5); ++w) dmax = part[w] > dmax ? part[w] : dmax;
        __syncthreads();
      }
      // Every thread owns a contiguous chunk [clo, chi) of the list for all passes of a reactivation, so the priority,
      // the exp() and the partial sums of its entries need no barrier in between; a reactivation costs four block
      // barriers (max / scan / owner / inhibition) instead of the dozen of a textbook block-wide sampler -- barrier
      // stalls were 4.6 warps per issued instruction in this kernel (profiles/r2_sfma_split_replay.txt).
      double lmax = 0.0;
#pragma unroll 1
      for (int j = clo; j < chi; ++j) {
        const uint32_t l = L[j];
        const int sp = l & 0xFFFF;
        const double cn = (mf & COBEL_SFMA_C_NORMALIZE) ? xdiv(Cc[j], cmax) : Cc[j];
        double r = xmul(xmul(cn, dvec(sp, Msc[j], cur, nxt)), xsub(1.0, I[sp]));    // C * D * (1 - I)
        if (r < thr) r = 0.0;
        R[j] = r;
        lmax = r > lmax ? r : lmax;
      }
      // block max (R >= 0): all-zero <=> np.sum(R) == 0 (sfma.py:316)
      for (int d = 16; d > 0; d >>= 1) { const double o = shfl_f64_xor(lmax, d); lmax = o > lmax ? o : lmax; }
      double* pmax = part + T + (it & 1) * 8;
      if (lane == 0) pmax[warp] = lmax;
      if (warp == 0 && !p.deterministic) {                                 // the draw is consumed only if a replay follows
        win.ensure(1, lane);
        const double u = win.peek(0);
        if (lane == 0) sh.u = u;
      }
      __syncthreads();                                                     // (1)
      double m = pmax[0];
      for (int w = 1; w < nw; ++w) m = pmax[w] > m ? pmax[w] : m;
      if (!(m > 0.0)) break;
      int jsel;
      if (p.deterministic) {                                               // argmax(R): first maximum
        if (tid == 0) sh.idx = 0x7fffffff;
        __syncthreads();
#pragma unroll 1
        for (int j = tid; j < nnz; j += T) if (R[j] == m) { atomicMin(&sh.idx, j); break; }
        __syncthreads();
        jsel = sh.idx;
        __syncthreads();
      } else {
        if (warp == 0) win.advance(1);
        // probs ~ exp(beta * R / max) - 1  (softmax(R, -1, beta), sfma.py:349-373); exp(0) - 1 == 0 exactly
        double local = 0.0;
#pragma unroll 1
        for (int j = clo; j < chi; ++j) {
          const double r = R[j];
          const double w = r > 0.0 ? xadd(exp(xmul((mf & COBEL_SFMA_R_RAW) ? r : xdiv(r, m), beta)), -1.0) : 0.0;
          R[j] = w;
          local += w;
        }
        // inverse-CDF draw (NumPy: searchsorted(cumsum(p) / cumsum(p)[-1], u, 'right')): exclusive scan of the
        // chunk sums, the first chunk whose running sum passes u * total owns the draw
        double inc = local;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const double o = shfl_f64_up(inc, d); if (lane >= d) inc += o; }
        double* psum = part + T + 16;
        if (lane == 31) psum[warp] = inc;
        __syncthreads();                                                   // (2)
        double off = 0.0, total = 0.0;
        for (int w = 0; w < nw; ++w) { if (w < warp) off += psum[w]; total += psum[w]; }
        const double excl = off + (inc - local);
        const double target = sh.u * total, tol = 1e-12 * total;
        const unsigned pass = __ballot_sync(kFull, local > 0.0 && excl + local > target);
        int* pc = reinterpret_cast<int*>(part + T + 24);
        if (lane == 0) pc[warp] = pass ? warp * 32 + __ffs(pass) - 1 : 0x7fffffff;
        part[tid] = excl;
        __syncthreads();                                                   // (3)
        int owner = pc[0];
        for (int w = 1; w < nw; ++w) owner = pc[w] < owner ? pc[w] : owner;
        bool near = false;
        if (owner == 0x7fffffff) {                                         // u * total rounded up to the total: the last positive weight
          jsel = nnz - 1;
          while (jsel > 0 && !(R[jsel] > 0.0)) --jsel;
          near = true;
        } else {                                                           // every thread walks the owner's chunk (broadcast reads)
          const int olo = owner * chunk < nnz ? owner * chunk : nnz, ohi = olo + chunk < nnz ? olo + chunk : nnz;
          double acc = part[owner];
          int found = -1, lastpos = olo;
          near = fabs(acc - target) < tol;
#pragma unroll 1
          for (int i = olo; i < ohi; ++i) {
            const double w = R[i];
            if (!(w > 0.0)) continue;
            lastpos = i;
            acc += w;
            if (fabs(acc - target) < tol) near = true;
            if (found < 0 && acc > target) found = i;
          }
          jsel = found >= 0 ? found : lastpos;
          if (found < 0) near = true;
        }
        if (near) flags |= COBEL_FLAG_CDF_NEAR_TIE;
      }
      const uint32_t l = L[jsel];
      action = l >> 16;
      cur = l & 0xFFFF;
      nxt = Msc[jsel];
#pragma unroll 1
      for (int s = tid; s < S; s += T) {                                   // sfma.py:333-335
        double v = xmul(I[s], dinh);
        if (s == cur) { v = xadd(v, p.i_step); v = v < 1.0 ? v : 1.0; }
        I[s] = v;
      }
      if (tid == 0) rep[count] = action * S + cur;
      ++count;
      __syncthreads();
    }
    log_replay(count);
    apply_batch(count);
    __syncthreads();
  }

  // M.I survives the replay (the next one resets it); M.T is zeroed after a trial with replay by the host side
  if (!random_path) {
#pragma unroll 1
    for (int e = tid; e < S; e += T) p.I[(size_t)n * S + e] = I[e];
  }
  flags = __syncthreads_or(flags);
  if (tid == 0) {
    p.stream.draw_count[n] = (int64_t)win.position();
    tr.n_replay[n] += nrep - nrep0;
    carry[2] = nrep; carry[3] = ncalls;
    if (tr.flags && flags) tr.flags[n] |= flags;
    if (p.td_acc) p.td_acc[n] = tdacc;
  }
}

// MODS = the memory's strength-modulation / normalisation switches (mod_flags) may be set; the common case
// (none) gets an instantiation without that code.
template <int A, bool MODS>
__global__ void __launch_bounds__(256) sfma_kernel(const __grid_constant__ CobelSFMAParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ BlockShared sh;
  const int S = p.world.n_states, K = p.world.n_starts, N = S * A, B = p.batch;
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int64_t n = blockIdx.x;
  const bool recency = p.recency != 0;
  // M.T is only read by the replay when `recency` is set, and it is zeroed after every trial with
  // replay (agent/sfma.py:324); it has to be tracked only if it is read or survives the trial
  const bool track_t = recency || p.no_replay != 0;
  const SfmaSmem so(S, A, T, B, track_t, p.random_replay != 0);
  double* Q = reinterpret_cast<double*>(smem + so.q);        // [s][a]
  double* Mr = reinterpret_cast<double*>(smem + so.mr);      // [s][a]
  double* C = reinterpret_cast<double*>(smem + so.c);        // [a*S + s]
  double* Tr = reinterpret_cast<double*>(smem + so.t);       // [a*S + s] (only when recency)
  double* R = reinterpret_cast<double*>(smem + so.r);        // scratch [a*S + s]
  double* I = reinterpret_cast<double*>(smem + so.inh);      // [s]
  double* part = reinterpret_cast<double*>(smem + so.part);
  int32_t* rep = reinterpret_cast<int32_t*>(smem + so.rep);  // reactivated flat indices of one replay
  uint16_t* Mx = reinterpret_cast<uint16_t*>(smem + so.mx);  // [s][a] next state | non-terminal << 15
  uint8_t* mbits = smem + so.mbits;                          // [s] valid-action bits
  double* cdft = reinterpret_cast<double*>(smem + so.cdf);   // random replay: m-fold sums of fl(1/n_valid)
  uint32_t* L = reinterpret_cast<uint32_t*>(smem + so.lst);  // experienced experiences (C > 0): action << 16 | state, ascending flat index
  // dependency scratch of the level-parallel batch aliases the (then idle) priority scratch
  uint32_t* wm = reinterpret_cast<uint32_t*>(R);
  uint32_t* rm = wm + S;

  const size_t g0 = (size_t)n * N;
  const uint8_t* amask = p.action_mask ? p.action_mask + n * p.mask_agent_stride : nullptr;
#pragma unroll 1
  for (int e = tid; e < N; e += T) {
    Q[e] = p.Q[g0 + e];
    Mr[e] = p.Mr[g0 + e];
    Mx[e] = (uint16_t)(p.Ms[g0 + e] | ((p.Mt[g0 + e] ? 1 : 0) << 15));
    C[e] = p.C[g0 + e];
    if (track_t) Tr[e] = p.T[g0 + e];
  }
#pragma unroll 1
  for (int e = tid; e < S; e += T) {
    I[e] = p.I[(size_t)n * S + e];
    uint32_t mb = (1u << A) - 1u;
    if (amask) {
      mb = 0;
      for (int a = 0; a < A; ++a) mb |= (amask[e * A + a] ? 1u : 0u) << a;
    }
    mbits[e] = (uint8_t)mb;
  }
  __syncthreads();

  // agent.random: batches are drawn uniformly over the unmasked experiences (retrieve_random_batch,
  // memory/sfma.py:375-416): probs = mask / sum(mask); NumPy's choice() searches u in
  // cumsum(probs) / cumsum(probs)[-1], i.e. in the m-fold sequential sums of fl(1 / n_valid)
  int nvalid = 0;
  if (p.random_replay) {
    if (tid == 0) {
      int m = 0;
      for (int a = 0; a < A; ++a)
        for (int sp = 0; sp < S; ++sp)
          if (mbits[sp] >> a & 1) ++m;
      const double pv = xdiv(1.0, int_to_f64(m));
      double c = 0.0;
      for (int j = 0; j < m; ++j) { c = xadd(c, pv); cdft[j] = c; }
      sh.idx = m;
    }
    __syncthreads();
    nvalid = sh.idx;
    __syncthreads();
  }

  DrawWindow win; win.init(p.stream, n, (uint64_t)p.stream.draw_count[n]);      // used by warp 0 only
  const double lr = p.lr[n], gamma = p.gamma[n], mlr = p.mem_lr[n];
  PolicyTab pt; pt.init(p.policy.kind, p.policy.param[n], lane);
  const bool learn = p.learn != 0;
  const bool masked = amask != nullptr;
  const bool do_replay = learn && !p.no_replay;
  const double beta = p.beta, thr = p.threshold, dinh = p.decay_inhibition, dstr = p.decay_strength, drec = p.decay_recency;
  const CobelTrace& tr = p.trace;
  int64_t nsteps = 0, nrep = 0, ncalls = 0;
  int flags = 0;
  const double* D = p.D;
  int mode = p.mode;                   // CTA-uniform; re-chosen per trial when agent.dynamic is set
  const int mf = MODS ? p.mod_flags : 0;   // COBEL_SFMA_MOD_* / *_NORMALIZE switches
  double cmax = 1.0, dmax = 1.0;       // np.amax(C) / np.amax(D[current_state]) when C_normalize / D_normalize
  double tdacc = p.td_acc ? p.td_acc[n] : 0.0;   // agent.td (maintained by warp 0)

  // agent.td += |td| for a batch of replayed updates, in replay order (agent/sfma.py:456); warp 0
  auto acc_td = [&](double tdl, bool active) {
    if (!p.td_acc) return;
    const unsigned act = __ballot_sync(kFull, active);
#pragma unroll 1
    for (int l = 0; l < 32 && (act >> l & 1u); ++l) tdacc = xadd(tdacc, fabs(shfl_f64(tdl, l)));
  };

  // similarity of experience i = (a, s') to the current experience, by replay mode
  // (memory/sfma.py:283-306)
  auto dvec = [&](int a, int sp, int cur, int nxt) -> double {
    const int ms = Mx[sp * A + a] & 0x7FFF;                 // states.flatten('F')[a*S + sp]
    const double* Dc = D + (size_t)cur * S;
    const double* Dn = D + (size_t)nxt * S;
    // D_normalize divides the current state's row by its maximum before the mode is applied (memory/sfma.py:286-288)
    auto dc = [&](int x) -> double { return (mf & COBEL_SFMA_D_NORMALIZE) ? xdiv(Dc[x], dmax) : Dc[x]; };
    switch (mode) {
      case MODE_FORWARD: return Dn[sp];
      case MODE_REVERSE: return dc(ms);
      case MODE_BLEND_FORWARD: return xadd(dc(sp), xmul(p.blend, Dn[sp]));
      case MODE_BLEND_REVERSE: return xadd(dc(sp), xmul(p.blend, dc(ms)));
      case MODE_INTERPOLATE: return xadd(xmul(p.interp_fwd, Dn[sp]), xmul(p.interp_rev, dc(ms)));
      case MODE_SWEEPING: return Dn[ms];
      default: return dc(sp);
    }
  };

  // SFMAMemory.replay (memory/sfma.py:238-347) + the Q updates of SFMA.replay (agent/sfma.py:416-419)
  auto replay = [&](int last, bool apply_updates) {
    if (p.random_replay && apply_updates) {
      // lane b of warp 0 resolves draw b: smallest m with cdf_m / cdf_last > u, then the m-th valid (a, s)
      if (warp == 0) {
        const double tot = cdft[nvalid - 1];
#pragma unroll 1
        for (int b0 = 0; b0 < B; b0 += 32) {
          const int nb = B - b0 < 32 ? B - b0 : 32;
          win.ensure(nb, lane);
          const double u = win.peek(lane < nb ? lane : 0);
          win.advance(nb);
          if (lane < nb) {
            int lo = 0, hi = nvalid - 1;                       // invariant: answer in [lo, hi]
            while (lo < hi) {
              const int mid = (lo + hi) >> 1;
              if (xdiv(cdft[mid], tot) > u) hi = mid; else lo = mid + 1;
            }
            int m = lo, e = -1;                                // m-th valid experience in F order
            for (int a = 0; a < A && e < 0; ++a)
              for (int sp = 0; sp < S; ++sp)
                if ((mbits[sp] >> a & 1) && m-- == 0) { e = a * S + sp; break; }
            rep[b0 + lane] = e;
          }
        }
      }
      __syncthreads();
      const int count = B;
      if (tr.replay_idx)
#pragma unroll 1
        for (int j = tid; j < count; j += T) {
          if (nrep + j < tr.replay_cap) tr.replay_idx[n * tr.replay_cap + nrep + j] = rep[j];
          else flags |= COBEL_FLAG_TRACE_OVERFLOW;
        }
#pragma unroll 1
      for (int e = tid; e < 2 * S; e += T) wm[e] = 0;
      __syncthreads();
      if (warp == 0) {
#pragma unroll 1
        for (int b0 = 0; b0 < count; b0 += 32) {
          const bool active = b0 + lane < count;
          int es = 0, ea = 0, es2 = 0, ent = 0;
          double er = 0.0;
          if (active) {
            const int e = rep[b0 + lane];
            ea = e / S; es = e - ea * S;
            er = Mr[es * A + ea];
            const uint16_t v = Mx[es * A + ea];
            es2 = v & 0x7FFF; ent = v >> 15;
          }
          double tdl = 0.0;
          td_batch_level_parallel<A>(Q, wm, rm, S, lane, active, es, ea, er, es2, ent, lr, gamma,
                                     masked ? mbits : nullptr, &tdl);
          acc_td(tdl, active);
        }
      }
      if (tr.replay_len && tid == 0) {
        if (ncalls < tr.replay_calls_cap) tr.replay_len[n * tr.replay_calls_cap + ncalls] = count;
        else flags |= COBEL_FLAG_TRACE_OVERFLOW;
      }
      nrep += count;
      ++ncalls;
      __syncthreads();
      return;
    }
    if (warp == 0) {
      win.ensure(2, lane);
      const int act0 = draw_integer(win.next(), A);                        // sfma.py:264 (always drawn)
      double u = 0.0;
      if (last < 0) u = win.next();                                        // sfma.py:272
      if (lane == 0) { sh.action = act0; sh.u = u; }
    }
    __syncthreads();
    int cur = last, action = sh.action;
    // Experiences that were never stored have strength 0, hence priority 0 and weight exp(0) - 1 = 0:
    // they can never be drawn and add exact zeros to every sum.  All passes below therefore run
    // over the compact, index-ordered list L of experiences with C > 0 (C is constant during a replay).
    int nnz;
    {
      const int chunk = (N + T - 1) / T;
      const int lo = tid * chunk < N ? tid * chunk : N, hi = lo + chunk < N ? lo + chunk : N;
      int cnt = 0;
#pragma unroll 1
      for (int i = lo; i < hi; ++i) cnt += C[i] > 0.0 ? 1 : 0;
      int off = block_exclusive_scan_int(cnt, part, tid, T, nnz);
#pragma unroll 1
      for (int i = lo; i < hi; ++i)
        if (C[i] > 0.0) { const int a = i / S; L[off++] = ((uint32_t)a << 16) | (uint32_t)(i - a * S); }
    }
    __syncthreads();
    if (mf & COBEL_SFMA_C_NORMALIZE) {                                     // np.amax(C): C is constant during a replay
      double lm = -__longlong_as_double(0x7FF0000000000000ll);
#pragma unroll 1
      for (int e = tid; e < N; e += T) lm = C[e] > lm ? C[e] : lm;
      for (int d = 16; d > 0; d >>= 1) { const double o = shfl_f64_xor(lm, d); lm = o > lm ? o : lm; }
      if (lane == 0) part[warp] = lm;
      __syncthreads();
      cmax = part[0];
      for (int w = 1; w < (T >> 5); ++w) cmax = part[w] > cmax ? part[w] : cmax;
      __syncthreads();
    }
    if (cur < 0) {                                                         // start ~ clip(C, 0) / sum
#pragma unroll 1
      for (int j = tid; j < nnz; j += T) { const uint32_t l = L[j]; R[j] = C[(l >> 16) * S + (l & 0xFFFF)]; }
      __syncthreads();
      const uint32_t l = L[block_sample(R, nnz, sh.u, part, &sh, tid, T, flags)];
      cur = l & 0xFFFF; action = l >> 16;
    }
    int nxt = Mx[cur * A + action] & 0x7FFF;
#pragma unroll 1
    for (int e = tid; e < S; e += T) I[e] = 0.0;                           // sfma.py:277
    __syncthreads();
    int count = 0;
    for (int it = 0; it < B; ++it) {
      if (mf & COBEL_SFMA_D_NORMALIZE) {                                   // np.amax(D[current_state])
        const double* Dc = D + (size_t)cur * S;
        double lm = -__longlong_as_double(0x7FF0000000000000ll);
#pragma unroll 1
        for (int e = tid; e < S; e += T) lm = Dc[e] > lm ? Dc[e] : lm;
        for (int d = 16; d > 0; d >>= 1) { const double o = shfl_f64_xor(lm, d); lm = o > lm ? o : lm; }
        if (lane == 0) part[warp] = lm;
        __syncthreads();
        dmax = part[0];
        for (int w = 1; w < (T >> 5); ++w) dmax = part[w] > dmax ? part[w] : dmax;
        __syncthreads();
      }
      double lmax = 0.0;
#pragma unroll 1
      for (int j = tid; j < nnz; j += T) {
        const uint32_t l = L[j];
        const int a = l >> 16, sp = l & 0xFFFF, i = a * S + sp;
        const double cn = (mf & COBEL_SFMA_C_NORMALIZE) ? xdiv(C[i], cmax) : C[i];
        double r = xmul(xmul(cn, dvec(a, sp, cur, nxt)), xsub(1.0, I[sp]));    // C * D * (1 - I)
        if (recency) r = xmul(r, Tr[i]);
        if (r < thr) r = 0.0;
        R[j] = r;
        lmax = r > lmax ? r : lmax;
      }
      // block max (R >= 0): all-zero <=> np.sum(R) == 0 (sfma.py:316)
      for (int d = 16; d > 0; d >>= 1) { const double o = shfl_f64_xor(lmax, d); lmax = o > lmax ? o : lmax; }
      if (lane == 0) part[warp] = lmax;
      __syncthreads();
      double m = part[0];
      for (int w = 1; w < (T >> 5); ++w) m = part[w] > m ? part[w] : m;
      __syncthreads();
      if (!(m > 0.0)) break;
      int jsel;
      if (p.deterministic) {                                               // argmax(R): first maximum
        if (tid == 0) sh.idx = 0x7fffffff;
        __syncthreads();
#pragma unroll 1
        for (int j = tid; j < nnz; j += T) if (R[j] == m) { atomicMin(&sh.idx, j); break; }
        __syncthreads();
        jsel = sh.idx;
        __syncthreads();
      } else {
        // probs ~ exp(beta * R / max) - 1  (softmax(R, -1, beta), sfma.py:349-373); exp(0) - 1 == 0 exactly
#pragma unroll 1
        for (int j = tid; j < nnz; j += T) { const double r = R[j]; R[j] = r > 0.0 ? xadd(exp(xmul((mf & COBEL_SFMA_R_RAW) ? r : xdiv(r, m), beta)), -1.0) : 0.0; }
        if (warp == 0) {
          win.ensure(1, lane);
          const double u = win.next();
          if (lane == 0) sh.u = u;
        }
        __syncthreads();
        jsel = block_sample(R, nnz, sh.u, part, &sh, tid, T, flags);
      }
      const uint32_t l = L[jsel];
      action = l >> 16;
      cur = l & 0xFFFF;
      const int e = action * S + cur;
      nxt = Mx[cur * A + action] & 0x7FFF;
#pragma unroll 1
      for (int s = tid; s < S; s += T) {                                   // sfma.py:333-335
        double v = xmul(I[s], dinh);
        if (s == cur) { v = xadd(v, p.i_step); v = v < 1.0 ? v : 1.0; }
        I[s] = v;
      }
      if (tid == 0) rep[count] = e;
      ++count;
      __syncthreads();
    }
    // apply the reactivated experiences to Q in order (agent/sfma.py:416-419)
    if (tr.replay_idx)
#pragma unroll 1
      for (int j = tid; j < count; j += T) {
        if (nrep + j < tr.replay_cap) tr.replay_idx[n * tr.replay_cap + nrep + j] = rep[j];
        else flags |= COBEL_FLAG_TRACE_OVERFLOW;
      }
#pragma unroll 1
    for (int e = tid; e < 2 * S; e += T) wm[e] = 0;                        // wm, rm alias R
    __syncthreads();
    if (warp == 0 && apply_updates) {
#pragma unroll 1
      for (int b0 = 0; b0 < count; b0 += 32) {
        const bool active = b0 + lane < count;
        int es = 0, ea = 0, es2 = 0, ent = 0;
        double er = 0.0;
        if (active) {
          const int e = rep[b0 + lane];
          ea = e / S; es = e - ea * S;
          er = Mr[es * A + ea];
          const uint16_t v = Mx[es * A + ea];
          es2 = v & 0x7FFF; ent = v >> 15;
        }
        double tdl = 0.0;
        td_batch_level_parallel<A>(Q, wm, rm, S, lane, active, es, ea, er, es2, ent, lr, gamma,
                                   masked ? mbits : nullptr, &tdl);
        acc_td(tdl, active);
      }
    }
    if (tr.replay_len && tid == 0) {
      if (ncalls < tr.replay_calls_cap) tr.replay_len[n * tr.replay_calls_cap + ncalls] = count;
      else flags |= COBEL_FLAG_TRACE_OVERFLOW;
    }
    nrep += count;
    ++ncalls;
    __syncthreads();
  };

  for (int trial = 0; trial < p.trials; ++trial) {
    // ---- reset (+ optional replay at trial start, agent/sfma.py:272-275) ------------------------
    if (warp == 0) {
      win.ensure(2, lane);
      const int s0 = __ldg(p.world.starts + draw_integer(win.next(), K));
      if (lane == 0) sh.last = s0;
    }
    __syncthreads();
    int s = sh.last;
    __syncthreads();
    // the replay at trial start only generates a trace (memory call, agent/sfma.py:272-275): no Q updates
    // (it runs whenever agent.start_replay is set, also with no_replay=True, like the reference)
    if (learn && p.start_replay) replay(s, false);
    // ---- the online steps of the trial: warp 0, warp-uniform ---------------------------------
    if (warp == 0) {
      double treward = 0.0;
      int step = 0, last = -1;
      for (;; ++step) {
        win.ensure(2, lane);
        double row[A];
        load_row<A>(Q + s * A, row);
        const int a = select_action_warp<A>(row, mbits[s], pt, win.next(), lane);
        const int s2 = p.world.tp_off ? stochastic_successor(p.world, s * A + a, win.next()) : __ldg(p.world.succ + s * A + a);
        const double r = __ldg(p.world.reward + s2);
        const int end = __ldg(p.world.terminal + s2);
        const int nt = 1 - end;
        if (tr.step_sa && lane == 0) {
          if (nsteps < tr.step_cap) { tr.step_sa[n * tr.step_cap + nsteps] = s * A + a; if (tr.step_next) tr.step_next[n * tr.step_cap + nsteps] = s2; }
          else flags |= COBEL_FLAG_TRACE_OVERFLOW;
        }
        ++nsteps;
        if (learn) {
          // SFMAMemory.store (memory/sfma.py:206-215): EMA reward, next state, flag, strengths, recency
          if (dstr != 1.0) {
#pragma unroll 1
            for (int e = lane; e < N; e += 32) C[e] = xmul(C[e], dstr);
          }
          if (track_t) {
#pragma unroll 1
            for (int e = lane; e < N; e += 32) Tr[e] = xmul(Tr[e], drec);
          }
          const double m0 = Mr[s * A + a];
          const double m1 = xadd(m0, xmul(mlr, xsub(r, m0)));
          // SFMA.update_q (agent/sfma.py:423-458): max over the unmasked actions of s'
          double row2[A];
          load_row<A>(Q + s2 * A, row2);
          const uint32_t mb = mbits[s2];
          double mx = -__longlong_as_double(0x7FF0000000000000ll);
#pragma unroll
          for (int x = 0; x < A; ++x) mx = (mb >> x & 1u) ? xmax(mx, row2[x]) : mx;
          const double q = Q[s * A + a];
          double td = xadd(r, xmul(nt ? gamma : 0.0, mx));
          td = xsub(td, q);
          const double qn = xadd(q, xmul(lr, td));
          tdacc = xadd(tdacc, fabs(td));
          __syncwarp();
          if (lane == 0) {
            Mr[s * A + a] = m1;
            Mx[s * A + a] = (uint16_t)(s2 | (nt << 15));
            C[a * S + s] = xadd(C[a * S + s], p.c_step);
            if (track_t) Tr[a * S + s] = 1.0;
            Q[s * A + a] = qn;
          }
          __syncwarp();
          if (mf & (COBEL_SFMA_MOD_REWARD_LOCAL | COBEL_SFMA_MOD_REWARD | COBEL_SFMA_MOD_STATE)) {
            // strength modulation of SFMAMemory.store, in the reference's order (memory/sfma.py:216-236)
            if ((mf & COBEL_SFMA_MOD_REWARD_LOCAL) && lane == 0)
              C[a * S + s] = xadd(C[a * S + s], xmul(r, p.reward_modulation));
            __syncwarp();
            if (mf & COBEL_SFMA_MOD_REWARD) {
              const double* Ds = D + (size_t)s * S;
#pragma unroll 1
              for (int e = lane; e < N; e += 32) C[e] = xadd(C[e], xmul(xmul(r, Ds[e % S]), p.reward_modulation));
              __syncwarp();
            }
            if ((mf & COBEL_SFMA_MOD_STATE) && lane < A) C[lane * S + s] = xadd(C[lane * S + s], 1.0);
            __syncwarp();
          }
        }
        s = s2;
        treward = xadd(treward, r);
        if (end) last = s2;
        if (end || step + 1 == p.steps) break;
      }
      if (lane == 0) {
        tr.trial_steps[n * p.trials + trial] = step;
        tr.trial_reward[n * p.trials + trial] = treward;
        sh.last = last;
      }
    }
    __syncthreads();
    if (do_replay) {
      const int last = sh.last;
      if (p.dynamic) {
        // agent/sfma.py:311-318: p('reverse') = 1 / (1 + exp(-(5 td - 2))), one categorical draw over
        // [p, 1 - p] (cdf normalised by its last entry), the accumulator restarts
        if (warp == 0) {
          win.ensure(1, lane);
          const double u = win.next();
          const double pm = xdiv(1.0, xadd(1.0, exp(-xsub(xmul(tdacc, 5.0), 2.0))));
          const double c0 = xdiv(pm, xadd(pm, xsub(1.0, pm)));
          if (fabs(c0 - u) < 1e-12) flags |= COBEL_FLAG_CDF_NEAR_TIE;      // exp() is not NumPy's bit for bit
          tdacc = 0.0;
          if (lane == 0) sh.idx = c0 > u ? MODE_REVERSE : MODE_DEFAULT;
        }
        __syncthreads();
        mode = sh.idx;
        if (p.trial_mode && tid == 0) p.trial_mode[n * p.trials + trial] = mode;
        __syncthreads();
      }
      for (int rpl = 0; rpl < p.nb_replays; ++rpl) replay(last, true);
      if (track_t) {
#pragma unroll 1
        for (int e = tid; e < N; e += T) Tr[e] = 0.0;           // M.T.fill(0), agent/sfma.py:324
      }
      __syncthreads();
    }
  }

  __syncthreads();
  if (learn) {
#pragma unroll 1
    for (int e = tid; e < N; e += T) {
      p.Q[g0 + e] = Q[e];
      p.Mr[g0 + e] = Mr[e];
      p.Ms[g0 + e] = Mx[e] & 0x7FFF;
      p.Mt[g0 + e] = Mx[e] >> 15;
      p.C[g0 + e] = C[e];
      // without the recency option T is never read; it is zero after every trial with replay
      if (track_t) p.T[g0 + e] = Tr[e];
      else if (do_replay && p.trials > 0) p.T[g0 + e] = 0.0;
    }
#pragma unroll 1
    for (int e = tid; e < S; e += T) p.I[(size_t)n * S + e] = I[e];
  }
  flags = __syncthreads_or(flags);
  if (tid == 0) {
    p.stream.draw_count[n] = (int64_t)win.position();
    tr.n_steps[n] += nsteps;
    tr.n_replay[n] += nrep;
    if (tr.flags && flags) tr.flags[n] |= flags;
    if (p.td_acc) p.td_acc[n] = tdacc;
  }
}

// The replay kernel's CTA size for S*A experiences and the capacity of its list of experienced (s, a) at that size
template <int A>
int replay_plan(const CobelSFMAParams& p, int& threads, int& cap) {
  const int S = p.world.n_states, N = S * A;
  threads = N <= 128 ? 64 : N <= 4096 ? 128 : 256;
  cap = ReplaySmem::fit(S, A, threads, p.batch, p.random_replay != 0, kMaxSmem - 512);
  const ReplaySmem rso(S, A, threads, p.batch, p.random_replay != 0, cap);
  COBEL_REQUIRE(cap >= 1 && rso.bytes <= kMaxSmem, COBEL_EUNSUPPORTED,
                "SFMA replay of %d states x %d actions needs %d bytes of shared memory", S, A, rso.bytes);
  return COBEL_OK;
}

// One launch of the replay kernel: `threads` per agent, a list of ph.list_cap entries
template <int A>
int replay_launch(const CobelSFMAParams& p, SfmaPhase ph, int threads, cudaStream_t st) {
  const ReplaySmem so(p.world.n_states, A, threads, p.batch, p.random_replay != 0, ph.list_cap);
  return launch_kernel(sfma_replay_kernel<A>, (unsigned)p.n_agents, threads, so.bytes, st, p, ph);
}

template <int A>
int launch(const CobelSFMAParams& p, cudaStream_t st) {
  const int S = p.world.n_states, N = S * A;
  COBEL_REQUIRE(S <= 0x7FFF, COBEL_EUNSUPPORTED, "SFMA kernel supports at most 32767 states");
  const int T = N <= 128 ? 64 : N <= 512 ? 128 : 256;
  // Split path: per-step work that touches single table entries only (no decay of C, M.T neither read nor kept,
  // no strength modulation over all experiences)
  const bool track_t = p.recency != 0 || (p.learn && p.no_replay);
  const bool split = p.decay_strength == 1.0 && !track_t && !(p.mod_flags & COBEL_SFMA_MOD_REWARD);
  // (state spaces whose tables exceed shared memory run on the split path only: its step kernel works on the tables
  //  in HBM and its replay kernel stages just the list of experienced (s, a))
  if (split) {
    int TR, cap;
    if (int rc = replay_plan<A>(p, TR, cap)) return rc;
    COBEL_CUDA_OK(cudaFuncSetAttribute(sfma_replay_kernel<A>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    const unsigned grid_step = (unsigned)((p.n_agents + 63) / 64);
    auto step = [&](SfmaPhase ph) { return launch_kernel(sfma_step_kernel<A>, grid_step, 64, 0, st, p, ph); };
    // The list of experienced (s, a) of a replay holds at most what the agent had when the call started plus one new
    // pair per step taken since (A with state_mod): with the caller's bound (exp_bound) a launch stages that many entries instead of
    // S*A -- at C4 22 KB instead of 40 KB per agent, 8 instead of 5 resident CTAs per SM.
    // CTA size: the replay's passes run over that list -- a few hundred entries -- and every warp repeats the
    // block-wide combines, so a small CTA with more CTAs per SM wins (20x20, 65536 agents, lists of <= 800 entries:
    // 0.88 / 1.19 / 1.11 / 0.73 x 10^9 agent-steps/s with 32 / 64 / 128 / 256 threads): 64 threads up to 1024 entries.
    auto replay = [&](SfmaPhase ph) {
      int lc = cap;
      if (p.exp_bound > 0) {
        // (state_mod strengthens every action of the visited state: up to A new entries per step, memory/sfma.py:234-236)
        const long long per_step = (p.mod_flags & COBEL_SFMA_MOD_STATE) ? A : 1;
        const long long bound = (long long)p.exp_bound - 1 + (long long)(ph.trial + (ph.start_replay ? 0 : 1)) * p.steps * per_step;
        if (bound < lc) lc = bound < 1 ? 1 : (int)bound;
      }
      ph.list_cap = lc;
      return replay_launch<A>(p, ph, lc <= 1024 ? 64 : TR, st);
    };
    // SfmaPhase{init, reset, n_trials, trial, start_replay}
    if (!p.learn) return step(SfmaPhase{1, 1, p.trials, 0, 0, cap});     // test(): all trials in one launch
    for (int t = 0; t < p.trials; ++t) {
      if (p.start_replay) {                                      // agent/sfma.py:272-275: trace only, no Q updates
        if (int rc = step(SfmaPhase{t == 0, 1, 0, t, 0, cap})) return rc;
        if (int rc = replay(SfmaPhase{0, 0, 0, t, 1, cap})) return rc;
        if (int rc = step(SfmaPhase{0, 0, 1, t, 0, cap})) return rc;
      } else if (int rc = step(SfmaPhase{t == 0, 1, 1, t, 0, cap})) {
        return rc;
      }
      if (int rc = replay(SfmaPhase{0, 0, 0, t, 0, cap})) return rc;   // agent/sfma.py:300-324 (no_replay keeps M.T: fused path)
    }
    // M.T.fill(0) after every trial with replay (agent/sfma.py:324); M.T is not tracked on this path
    if (p.trials > 0) COBEL_CUDA_OK(cudaMemsetAsync(p.T, 0, (size_t)p.n_agents * N * sizeof(double), st));
    return COBEL_OK;
  }
  const SfmaSmem so(S, A, T, p.batch, p.recency != 0 || p.no_replay != 0, p.random_replay != 0);
  COBEL_REQUIRE(so.bytes <= kMaxSmem, COBEL_EUNSUPPORTED,
                "SFMA tables of %d states x %d actions need %d bytes of shared memory", S, A, so.bytes);
  return launch_kernel(p.mod_flags ? sfma_kernel<A, true> : sfma_kernel<A, false>, (unsigned)p.n_agents, T, so.bytes, st, p);
}

// SFMAMemory.replay(batch, state) / SFMA.replay(batch, state) as a stand-alone call: the replay kernel of the split path
template <int A>
int replay_only(const CobelSFMAParams& p, const int32_t* state, int apply_updates, cudaStream_t st) {
  COBEL_REQUIRE(p.world.n_states <= 0x7FFF, COBEL_EUNSUPPORTED, "SFMA kernel supports at most 32767 states");
  int T, cap;
  if (int rc = replay_plan<A>(p, T, cap)) return rc;
  if (int rc = cobel_set_carry(p.carry, 4, state, p.n_agents, st)) return rc;
  return replay_launch<A>(p, SfmaPhase{0, 0, 0, 0, apply_updates == 1 ? 0 : (apply_updates == 2 ? 2 : 1), cap}, T, st);
}

}  // namespace

extern "C" int cobel_sfma_run(const CobelSFMAParams* pp, void* stream) {
  COBEL_REQUIRE(pp != nullptr, COBEL_EINVAL, "null params");
  const CobelSFMAParams& p = *pp;
  int rc = cobel_validate_common(p.n_agents, p.world, p.stream, p.policy, p.trace, p.trials, p.steps);
  if (rc) return rc;
  COBEL_REQUIRE(p.Q && p.Mr && p.Ms && p.Mt && p.C && p.T && p.I && p.D && p.lr && p.gamma && p.mem_lr, COBEL_EINVAL,
                "agent tables missing");
  COBEL_REQUIRE(p.carry, COBEL_EINVAL, "carry scratch missing");
  COBEL_REQUIRE(p.batch >= 0 && p.nb_replays >= 0, COBEL_EINVAL, "batch and nb_replays must be >= 0");
  COBEL_REQUIRE(p.mode >= MODE_DEFAULT && p.mode <= MODE_SWEEPING, COBEL_EINVAL, "unknown replay mode %d", p.mode);
  if (p.trials == 0) return COBEL_OK;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  COBEL_DISPATCH_A(p.world.n_actions, return launch<A>(p, st));
}

extern "C" int cobel_sfma_replay(const CobelSFMAParams* pp, const int32_t* state, int apply_updates, void* stream) {
  COBEL_REQUIRE(pp != nullptr && state != nullptr, COBEL_EINVAL, "null params");
  const CobelSFMAParams& p = *pp;
  COBEL_REQUIRE(p.n_agents > 0 && p.stream.draw_count && p.trace.n_replay && p.trace.replay_idx && p.trace.replay_len && p.carry,
                COBEL_EINVAL, "cobel_sfma_replay needs the stream, trace.replay_idx / replay_len / n_replay and the carry scratch");
  COBEL_REQUIRE(p.Mr && p.Ms && p.Mt && p.C && p.I && p.D, COBEL_EINVAL, "memory tables missing");
  COBEL_REQUIRE(apply_updates != 1 || (p.Q && p.lr && p.gamma), COBEL_EINVAL, "Q / lr / gamma missing");
  COBEL_REQUIRE(p.batch >= 0 && p.nb_replays >= 0 && !p.recency, COBEL_EINVAL, "batch and nb_replays must be >= 0; recency runs inside train() only");
  COBEL_REQUIRE(p.mode >= MODE_DEFAULT && p.mode <= MODE_SWEEPING, COBEL_EINVAL, "unknown replay mode %d", p.mode);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  COBEL_DISPATCH_A(p.world.n_actions, return replay_only<A>(p, state, apply_updates, st));
}
