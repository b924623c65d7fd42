// dynaq.cu -- K1: the whole DynaQ.train()/test() loop of N independent agents in one launch.
//
// Reference: agent/dyna_q.py:140-330 (trial/step loop, update_q, replay),
// memory/dyna_q.py:62-157 (store, retrieve_batch), policy/greedy.py, policy/softmax.py,
// interface/gridworld.py:92-145.  Semantics: SURVEY.md Appendix A.4.
//
// Mapping: ONE WARP PER AGENT, agent tables resident in shared memory for the whole launch
// (HBM is touched once: coalesced stage-in / stage-out).  Per environment step the warp
//   * takes the step's 34 uniforms from the agent's stream window (one Philox block per lane per refill;
//     the PLAIN kernel keeps 256 draws in shared memory, i.e. seven steps per refill),
//   * selects the action and steps the environment warp-uniformly (PLAIN: tie-pattern CDF table),
//   * draws the 32 replay indices one per lane, gathers the 32 experiences in parallel and
//     applies the 32 TD updates in dependency levels (td_batch_level_parallel): one speculative
//     pass against the pre-batch table drops the updates that provably leave Q bit-identical
//     (80 % of the C2 batches are no-ops as a whole), the rest run in rounds of updates that do
//     not touch each other's rows, so the reference's strictly sequential 32-update chain
//     collapses to 0.66 rounds on average (5.3 without the pass) with bit-identical results.
// The PLAIN kernel reads the replay gather before the action selection (see its step loop).
// (v1 of this kernel used one thread per agent: 180 warp-instructions per update at one
//  instruction per 5 cycles, profiles/r1_dynaq_v1_thread_per_agent.txt.)
#include "warp_agent.cuh"

namespace {

constexpr int kWarpsPerCta = 4;

struct AgentSmem {      // byte offsets inside one agent's shared-memory block
  int q, mr, mx, wm, rm, ptab, draws, vmax, pat, bytes;
  // tables = false: Q / M stay in HBM (state spaces whose tables do not fit), only the dependency masks are on chip
  // sums = true: the row summaries V (S doubles) and P (S bytes) of the PLAIN kernel with A <= 4
  __host__ __device__ AgentSmem(int S, int A, bool plain, bool tables = true, bool sums = false) {
    const bool eps_tab = plain && A <= 4;
    const int SA = tables ? S * A : 0;
    q = 0;
    mr = q + SA * 8;
    wm = mr + SA * 8;
    rm = wm + S * 4;
    mx = rm + S * 4;
    ptab = (mx + SA * 2 + 15) & ~15;
    draws = ptab + (eps_tab ? kEpsTabDoubles * 8 : 0);
    vmax = draws + (plain ? kSmemDraws * 8 : 0);
    pat = vmax + (sums ? S * 8 : 0);
    bytes = sums ? (pat + S + 15) & ~15 : vmax;
  }
};

struct WorldSmem {      // byte offsets of the CTA-shared environment tables
  int rew, succ, starts, term, bytes;
  __host__ __device__ WorldSmem(int S, int A, int K) {
    rew = 0;
    succ = rew + S * 8;
    starts = succ + S * A * 4;
    term = starts + K * 4;
    bytes = (term + S + 15) & ~15;
  }
};

// PLAIN = the common production case (epsilon-greedy training with per-step replay, no optional trace buffers,
// no action mask, deterministic world): a kernel without the per-step checks and the other policies' code
// (the instruction count per step is what bounds this kernel).
// HBM = the agent's tables (and the environment's) are too large for shared memory: Q / M.rewards / M.states /
// M.terminals are read and written in place in HBM / L2 (a replay is 32 independent gathers per lane-parallel
// round, so the DRAM latency of a step is paid about six times, not 33), the world tables go through the read-only
// path, only the two dependency masks of the level-parallel replay (8 bytes per state) stay on chip.
// SUM (PLAIN, A <= 4): the agent keeps the row summaries V[s] = row_max(Q[s,:]) and P[s] = its tie pattern on chip
// (refresh_row_summary), so the action selection, the online update's target and the replay's speculative pass read
// one entry instead of a row and its maximum; a step that writes a row refreshes its summaries.
template <int A, bool PLAIN, bool HBM = false, bool SUM = false>
__global__ void __launch_bounds__(kWarpsPerCta * 32, HBM ? 1 : 7) dynaq_warp_kernel(const __grid_constant__ CobelDynaQParams p) {
  static_assert(!(PLAIN && HBM), "the HBM path is the generic kernel");
  static_assert(!SUM || (PLAIN && A <= 4), "row summaries go with the tie-pattern table");
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, K = p.world.n_starts, SA = S * A;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const WorldSmem wo(HBM ? 0 : S, A, HBM ? 0 : K);
  constexpr bool kEpsTab = PLAIN && A <= 4;      // tie-pattern CDF table instead of per-step probabilities
  const AgentSmem ao(S, A, PLAIN, !HBM, SUM);

  double* rew_s = reinterpret_cast<double*>(smem + wo.rew);
  int32_t* succ_s = reinterpret_cast<int32_t*>(smem + wo.succ);
  int32_t* starts_s = reinterpret_cast<int32_t*>(smem + wo.starts);
  uint8_t* term_s = smem + wo.term;
  if constexpr (!HBM) {
    for (int e = threadIdx.x; e < SA; e += blockDim.x) succ_s[e] = p.world.succ[e];
    for (int e = threadIdx.x; e < S; e += blockDim.x) { rew_s[e] = p.world.reward[e]; term_s[e] = p.world.terminal[e]; }
    for (int e = threadIdx.x; e < K; e += blockDim.x) starts_s[e] = p.world.starts[e];
    __syncthreads();
  }
  auto w_succ = [&](int sa) -> int { if constexpr (HBM) return __ldg(p.world.succ + sa); else return succ_s[sa]; };
  auto w_rew = [&](int x) -> double { if constexpr (HBM) return __ldg(p.world.reward + x); else return rew_s[x]; };
  auto w_term = [&](int x) -> int { if constexpr (HBM) return __ldg(p.world.terminal + x); else return term_s[x]; };
  auto w_start = [&](int k) -> int { if constexpr (HBM) return __ldg(p.world.starts + k); else return starts_s[k]; };

  const int64_t n = (int64_t)blockIdx.x * blockDim.x / 32 + warp;
  if (n >= p.n_agents) return;                      // whole warp leaves; no block-wide sync below

  unsigned char* blk = smem + wo.bytes + (size_t)warp * ao.bytes;
  const size_t g0 = (size_t)n * SA;
  double* Q = HBM ? p.Q + g0 : reinterpret_cast<double*>(blk + ao.q);
  double* Mr = HBM ? p.Mr + g0 : reinterpret_cast<double*>(blk + ao.mr);
  uint16_t* Mx = reinterpret_cast<uint16_t*>(blk + ao.mx);     // next state | non-terminal << 15 (on-chip tables)
  int32_t* Msg = p.Ms + g0;                                    // (HBM tables)
  int32_t* Mtg = p.Mt + g0;
  uint32_t* wm = reinterpret_cast<uint32_t*>(blk + ao.wm);
  uint32_t* rm = reinterpret_cast<uint32_t*>(blk + ao.rm);
  auto m_next = [&](int i, int& s2, int& nt) {
    if constexpr (HBM) { s2 = Msg[i]; nt = Mtg[i] ? 1 : 0; }
    else { const uint16_t v = Mx[i]; s2 = v & 0x7FFF; nt = v >> 15; }
  };
  auto m_set = [&](int i, int s2, int nt) {
    if constexpr (HBM) { Msg[i] = s2; Mtg[i] = nt; }
    else Mx[i] = (uint16_t)(s2 | (nt << 15));
  };

  if constexpr (!HBM) {
    for (int e = lane; e < SA; e += 32) {
      Q[e] = p.Q[g0 + e];
      Mr[e] = p.Mr[g0 + e];
      Mx[e] = (uint16_t)(p.Ms[g0 + e] | ((p.Mt[g0 + e] ? 1 : 0) << 15));
    }
  }
  __syncwarp();

  for (int e = lane; e < S; e += 32) { wm[e] = 0; rm[e] = 0; }
  double* V = reinterpret_cast<double*>(blk + ao.vmax);
  uint8_t* P = blk + ao.pat;
  if constexpr (SUM)      // from the staged Q, which may hold any values (ties, -0.0); eps_cdf_table_init syncs
    for (int e = lane; e < S; e += 32) refresh_row_summary<A>(Q, V, P, e);
  typename WindowFor<PLAIN>::type win; win.init(p.stream, n, (uint64_t)p.stream.draw_count[n]);
  win.attach(reinterpret_cast<double*>(blk + ao.draws));
  const double lr = p.lr[n], gamma = p.gamma[n], mlr = p.mem_lr[n];
  PolicyTab pt; pt.init(p.policy.kind, p.policy.param[n], lane);
  double* ptab = reinterpret_cast<double*>(blk + ao.ptab);
  if constexpr (kEpsTab) eps_cdf_table_init<A>(ptab, pt, lane);
  const uint8_t* amask = (!PLAIN && p.action_mask) ? p.action_mask + n * p.mask_agent_stride : nullptr;
  const int B = PLAIN ? 32 : p.batch;           // the PLAIN kernel is built for the reference's default batch of 32
  const bool learn = PLAIN || p.learn != 0;
  const bool step_replay = PLAIN || (learn && !p.no_replay && !p.episodic_replay);   // a batch of 0 is still a (draw-free) call
  const bool trial_replay = !PLAIN && learn && !p.no_replay && p.episodic_replay;
  const CobelTrace& tr = p.trace;
  int64_t nsteps = 0, nrep = 0, ncalls = 0;
  int flags = 0;

  // memory/dyna_q.py:137-157 + agent/dyna_q.py:329-330: B uniform draws over S*A (C-order
  // unravel), applied in order; 32 at a time, one per lane.
  auto replay = [&]() {
    for (int b0 = 0; b0 < B; b0 += 32) {
      const int nb = B - b0 < 32 ? B - b0 : 32;
      win.ensure(nb, lane);
      const bool active = lane < nb;
      const double u = win.peek(active ? lane : 0);
      win.advance(nb);
      int rs = 0, ra = 0, rs2 = 0, rnt = 0;
      double rr = 0.0;
      if (active) {
        const int i = draw_integer(u, SA);
        rs = i / A; ra = i - rs * A;
        rr = Mr[i];
        m_next(i, rs2, rnt);
        if (!PLAIN && tr.replay_idx) {
          if (nrep + lane < tr.replay_cap) tr.replay_idx[n * tr.replay_cap + nrep + lane] = i;
          else flags |= COBEL_FLAG_TRACE_OVERFLOW;
        }
      }
      td_batch_level_parallel<A>(Q, wm, rm, S, lane, active, rs, ra, rr, rs2, rnt, lr, gamma);
      nrep += nb;
    }
    if (!PLAIN && tr.replay_len && lane == 0) {
      if (ncalls < tr.replay_calls_cap) tr.replay_len[n * tr.replay_calls_cap + ncalls] = B;
      else flags |= COBEL_FLAG_TRACE_OVERFLOW;
    }
    ++ncalls;
  };

  for (int trial = 0; trial < p.trials; ++trial) {
    // interface/gridworld.py:142: one uniform draw over the starting states
    win.ensure(3 + (step_replay && B <= 32 ? B : 0), lane);
    int s = w_start(draw_integer(win.next(), K));
    double treward = 0.0;
    int step = 0;
    if constexpr (PLAIN) {
      // The replay gather (index, Mr, Mx) depends on the window and M only, not on the step's action: it is read
      // before the action selection and the store, so its shared-memory latency overlaps theirs, and the lane whose
      // index is the stored (s,a) takes the stored values -- what the sequential order reads.
      for (;; ++step) {
        win.ensure(34, lane);
        const int i = draw_integer(win.peek(1 + lane), SA);
        double rr = Mr[i];
        int rs2, rnt;
        m_next(i, rs2, rnt);
        int a;
        if constexpr (SUM) {
          a = select_action_eps_pattern<A>(P[s], ptab, win.next(), lane);
        } else {
          double row[A];
          load_row<A>(Q + s * A, row);
          if constexpr (kEpsTab) a = select_action_eps_tab<A>(row, ptab, win.next(), lane);
          else a = select_action_warp<A, COBEL_POLICY_EPS_GREEDY>(row, (1u << A) - 1u, pt, win.next(), lane);
        }
        const int sa = s * A + a;
        const int s2 = w_succ(sa);
        const double r = w_rew(s2);
        const int end = w_term(s2);
        const int nt = 1 - end;
        // memory/dyna_q.py:92-96 (store first), then agent/dyna_q.py:275-301 (online update)
        const double m0 = Mr[sa];
        const double m1 = xadd(m0, xmul(mlr, xsub(r, m0)));
        double row2[A];
        if constexpr (!SUM) load_row<A>(Q + s2 * A, row2);
        const double q = Q[sa];
        const double g = nt ? gamma : 0.0;
        // SUM: s2 == s reads V[s] before the write below, as the sequential update reads the row before its write
        double td = xadd(r, xmul(g, SUM ? V[s2] : row_max<A>(row2)));
        td = xsub(td, q);
        const double qn = xadd(q, xmul(lr, td));
        if (i == sa) { rr = m1; rs2 = s2; rnt = nt; }
        const int rs = i / A, ra = i - rs * A;
        __syncwarp();
        if (lane == 0) {
          Mr[sa] = m1;
          m_set(sa, s2, nt);
          Q[sa] = qn;
          // warp-uniform: 7 % of C2's online updates change Q[s,a]
          if (SUM && __double_as_longlong(qn) != __double_as_longlong(q)) refresh_row_summary<A>(Q, V, P, s);
        }
        __syncwarp();
        td_batch_level_parallel<A, SUM>(Q, wm, rm, S, lane, true, rs, ra, rr, rs2, rnt, lr, gamma, nullptr, nullptr, V, P);
        win.advance(32);
        ++nsteps;
        treward = xadd(treward, r);
        if (end || step + 1 == p.steps) break;
        s = s2;
      }
    } else for (;; ++step) {
      win.ensure(2 + (step_replay && B <= 32 ? B : 0), lane);
      double row[A];
      load_row<A>(Q + s * A, row);
      uint32_t mask = (1u << A) - 1u;
      if (amask) {
        mask = 0;
#pragma unroll
        for (int a = 0; a < A; ++a) mask |= (amask[s * A + a] ? 1u : 0u) << a;
      }
      const int a = select_action_warp<A>(row, mask, pt, win.next(), lane);
      const int s2 = p.world.tp_off ? stochastic_successor(p.world, s * A + a, win.next()) : w_succ(s * A + a);
      const double r = w_rew(s2);
      const int end = w_term(s2);
      const int nt = 1 - end;
      if (tr.step_sa && lane == 0) {
        if (nsteps < tr.step_cap) { tr.step_sa[n * tr.step_cap + nsteps] = s * A + a; if (tr.step_next) tr.step_next[n * tr.step_cap + nsteps] = s2; }
        else flags |= COBEL_FLAG_TRACE_OVERFLOW;
      }
      ++nsteps;
      if (learn) {
        // memory/dyna_q.py:92-96 (store first), then agent/dyna_q.py:275-301 (online update);
        // every lane computes the same values, lane 0 commits them
        const double m0 = Mr[s * A + a];
        const double m1 = xadd(m0, xmul(mlr, xsub(r, m0)));
        double row2[A];
        load_row<A>(Q + s2 * A, row2);
        const double q = Q[s * A + a];
        const double g = nt ? gamma : 0.0;
        double td = xadd(r, xmul(g, row_max<A>(row2)));
        td = xsub(td, q);
        const double qn = xadd(q, xmul(lr, td));
        if (tr.step_td && lane == 0) {               // the step's slot of step_sa (nsteps already counts it)
          if (nsteps <= tr.step_cap) tr.step_td[n * tr.step_cap + nsteps - 1] = td;
          else flags |= COBEL_FLAG_TRACE_OVERFLOW;
        }
        __syncwarp();
        if (lane == 0) {
          Mr[s * A + a] = m1;
          m_set(s * A + a, s2, nt);
          Q[s * A + a] = qn;
        }
        __syncwarp();
      }
      s = s2;
      if (step_replay) replay();
      treward = xadd(treward, r);
      if (end || step + 1 == p.steps) break;
    }
    if (lane == 0) {                                 // logs['steps'] = index of the last step
      tr.trial_steps[n * p.trials + trial] = step;
      tr.trial_reward[n * p.trials + trial] = treward;
    }
    if (trial_replay) replay();
  }

  __syncwarp();
  if (learn && !HBM) {
    for (int e = lane; e < SA; e += 32) {
      p.Q[g0 + e] = Q[e];
      p.Mr[g0 + e] = Mr[e];
      p.Ms[g0 + e] = Mx[e] & 0x7FFF;
      p.Mt[g0 + e] = Mx[e] >> 15;
    }
  }
  flags = __reduce_or_sync(kFull, flags);
  if (lane == 0) {
    p.stream.draw_count[n] = (int64_t)win.position();
    tr.n_steps[n] += nsteps;
    tr.n_replay[n] += PLAIN ? nsteps * 32 : nrep;
    if (tr.flags && flags) tr.flags[n] |= flags;
  }
}


// ---------------------------------------------------------------------------
// dynaq_pair_kernel: the PLAIN case with TWO AGENTS PER WARP (16 lanes each), A <= 4.
// The online part of a step (action selection, environment step, store, online update, stream refill) is
// warp-uniform work: with one agent per warp all 32 lanes repeat it, 151 of the 389 warp-instructions of an
// agent-step (profiles/r1_dynaq_v7_plain.txt).  Here each half-warp runs its own agent -- own trial / step
// counters, own tables, own stream -- so that work is issued once per two agents, and the replay batch of 32 is
// applied as two level-parallel passes of 16 (lane = update; the passes of the two agents share the rounds).
// The level-parallel routine is the one of the warp-per-agent kernel: its dependency masks live in per-agent
// arrays and hold warp lane bits, so the two halves never see each other.
// Stream: a ring of 128 draws per agent in shared memory, refilled 32 draws at a time (one Philox block per lane
// of the half) whenever fewer than a step's 34 are left -- every generated draw is consumed.
// ---------------------------------------------------------------------------
constexpr int kPairWarps = 2;          // warps per CTA (4 agents)
constexpr int kRing = 128;             // draws in an agent's ring

struct PairSmem {       // byte offsets inside one agent's shared-memory block
  int q, mr, mx, wm, rm, ptab, ring, bytes;
  __host__ __device__ PairSmem(int S, int A) {
    const int SA = S * A;
    q = 0;
    mr = q + SA * 8;
    wm = mr + SA * 8;
    rm = wm + S * 4;
    mx = rm + S * 4;
    ptab = (mx + SA * 2 + 15) & ~15;
    ring = ptab + kEpsTabDoubles * 8;
    bytes = ring + kRing * 8;
  }
};

template <int A>
__global__ void __launch_bounds__(kPairWarps * 32, 14) dynaq_pair_kernel(const __grid_constant__ CobelDynaQParams p) {
  static_assert(A <= 4, "tie-pattern table");
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, K = p.world.n_starts, SA = S * A;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, half = lane >> 4, h = lane & 15;
  const WorldSmem wo(S, A, K);
  const PairSmem ao(S, A);
  double* rew_s = reinterpret_cast<double*>(smem + wo.rew);
  int32_t* succ_s = reinterpret_cast<int32_t*>(smem + wo.succ);
  int32_t* starts_s = reinterpret_cast<int32_t*>(smem + wo.starts);
  uint8_t* term_s = smem + wo.term;
  for (int e = threadIdx.x; e < SA; e += blockDim.x) succ_s[e] = p.world.succ[e];
  for (int e = threadIdx.x; e < S; e += blockDim.x) { rew_s[e] = p.world.reward[e]; term_s[e] = p.world.terminal[e]; }
  for (int e = threadIdx.x; e < K; e += blockDim.x) starts_s[e] = p.world.starts[e];
  __syncthreads();

  const int64_t n = ((int64_t)blockIdx.x * kPairWarps + warp) * 2 + half;
  const bool mine = n < p.n_agents;                   // a half without an agent idles on zeroed tables
  const int64_t nn = mine ? n : p.n_agents - 1;
  unsigned char* blk = smem + wo.bytes + (size_t)(warp * 2 + half) * ao.bytes;
  const size_t g0 = (size_t)nn * SA;
  double* Q = reinterpret_cast<double*>(blk + ao.q);
  double* Mr = reinterpret_cast<double*>(blk + ao.mr);
  uint16_t* Mx = reinterpret_cast<uint16_t*>(blk + ao.mx);     // next state | non-terminal << 15
  uint32_t* wm = reinterpret_cast<uint32_t*>(blk + ao.wm);
  uint32_t* rm = reinterpret_cast<uint32_t*>(blk + ao.rm);
  double* ptab = reinterpret_cast<double*>(blk + ao.ptab);
  double* ring = reinterpret_cast<double*>(blk + ao.ring);
  for (int e = h; e < SA; e += 16) {
    Q[e] = mine ? p.Q[g0 + e] : 0.0;
    Mr[e] = mine ? p.Mr[g0 + e] : 0.0;
    Mx[e] = mine ? (uint16_t)(p.Ms[g0 + e] | ((p.Mt[g0 + e] ? 1 : 0) << 15)) : (uint16_t)0;
  }
  for (int e = h; e < S; e += 16) { wm[e] = 0; rm[e] = 0; }
  for (int e = h; e < kRing; e += 16) ring[e] = 0.0;
  const double lr = p.lr[nn], gamma = p.gamma[nn], mlr = p.mem_lr[nn];
  {
    // the agent's 2^A - 1 normalised CDFs by tie pattern (see eps_cdf_table_init): lane h = pattern h
    const double eps = p.policy.param[nn];
    const int pat = h & ((1 << A) - 1), k = __popc(pat);
    const double base = xdiv(eps, (double)A);
    const double tie = xdiv(xsub(1.0, eps), (double)(k > 0 ? k : 1));
    const double top = xadd(base, tie), low = xadd(base, 0.0);
    double cdf[A];
    double c = (pat & 1) ? top : low;
    cdf[0] = c;
#pragma unroll
    for (int a = 1; a < A; ++a) { c = xadd(c, (pat >> a & 1) ? top : low); cdf[a] = c; }
    if (c != 1.0) {
#pragma unroll
      for (int a = 0; a < A; ++a) cdf[a] = xdiv(cdf[a], c);
    }
    if (h > 0 && h < (1 << A)) {
#pragma unroll
      for (int a = 0; a < 4; ++a) ptab[pat * 4 + a] = a < A ? cdf[a] : 2.0;
    }
  }
  // stream state of the half: the ring holds draws [gen - 128, gen), the next draw is gen - avail
  const uint64_t agent = (uint64_t)(p.stream.agent_id_base + nn);
  const uint32_t key0 = (uint32_t)p.stream.seed, key1 = (uint32_t)(p.stream.seed >> 32);
  const uint64_t pos0 = (uint64_t)p.stream.draw_count[nn];
  uint64_t gblk = (pos0 & ~31ull) >> 1;               // Philox block of ring slot wr
  int wr = 0;                                         // ring slot that the next refill writes (multiple of 32)
  int rd = (int)(pos0 & 31ull);                       // ring slot of the next draw
  int avail = -rd;                                    // generated draws not yet consumed
  const CobelTrace& tr = p.trace;
  bool live = mine && p.trials > 0;
  bool fresh = true;                                  // the next step starts a trial
  int s = 0, step = 0, trial = 0;
  int nsteps = 0;
  double treward = 0.0;
  __syncwarp();

  while (__any_sync(kFull, live)) {
    // ---- stream: at least one step's draws (reset + action + 32 replay indices) ----
    for (;;) {
      const bool need = live && avail < 34;
      if (!__any_sync(kFull, need)) break;
      const uint64_t b = gblk + (uint64_t)h;
      uint32_t o[4];
      philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), (uint32_t)agent, (uint32_t)(agent >> 32), key0, key1, o);
      if (need) {
        reinterpret_cast<double2*>(ring)[(wr >> 1) + h] = make_double2(u53(o[0], o[1]), u53(o[2], o[3]));
        gblk += 16; wr = (wr + 32) & (kRing - 1); avail += 32;
      }
    }
    __syncwarp();
    // ---- interface/gridworld.py:142 (reset), policy, environment ----
    if (fresh) {
      if (live) { s = starts_s[draw_integer(ring[rd], K)]; rd = (rd + 1) & (kRing - 1); --avail; }
      fresh = false; step = 0; treward = 0.0;
    }
    double row[A];
    load_row<A>(Q + s * A, row);
    const double ua = ring[rd];
    int a;
    {
      const double m = row_max<A>(row);
      uint32_t ties = 0;
#pragma unroll
      for (int x = 0; x < A; ++x) ties |= (row[x] == m ? 1u : 0u) << x;
      const double edge = ptab[ties * 4 + (h & 3)];
      const unsigned bal = __ballot_sync(kFull, h < A - 1 && edge <= ua);
      a = __popc((bal >> (half * 16)) & 0xFFFFu);
    }
    const int sa = s * A + a;
    const int s2 = succ_s[sa];
    const double r = rew_s[s2];
    const int end = term_s[s2];
    const int nt = 1 - end;
    {
      // memory/dyna_q.py:92-96 (store first), then agent/dyna_q.py:275-301 (online update)
      const double m0 = Mr[sa];
      const double m1 = xadd(m0, xmul(mlr, xsub(r, m0)));
      double row2[A];
      load_row<A>(Q + s2 * A, row2);
      const double q = Q[sa];
      const double g = nt ? gamma : 0.0;
      double td = xadd(r, xmul(g, row_max<A>(row2)));
      td = xsub(td, q);
      const double qn = xadd(q, xmul(lr, td));
      __syncwarp();
      if (live && h == 0) {
        Mr[sa] = m1;
        Mx[sa] = (uint16_t)(s2 | (nt << 15));
        Q[sa] = qn;
      }
      __syncwarp();
    }
    // ---- replay: memory/dyna_q.py:137-157 + agent/dyna_q.py:329-330, 32 updates as two passes of 16 ----
#pragma unroll 1
    for (int b0 = 0; b0 < 32; b0 += 16) {
      const double u = ring[(rd + 1 + b0 + h) & (kRing - 1)];
      const int i = draw_integer(u, SA);
      const int rs = i / A, ra = i - rs * A;
      const double rr = Mr[i];
      const uint16_t v = Mx[i];
      td_batch_level_parallel<A>(Q, wm, rm, S, lane, live, rs, ra, rr, v & 0x7FFF, v >> 15, lr, gamma);
    }
    // ---- bookkeeping of the half, branch-free (the two halves end their trials at different steps) ----
    {
      const bool fin = end || step + 1 == p.steps;
      const double tw = xadd(treward, r);
      if (live && fin && h == 0) {                       // logs['steps'] = index of the last step
        tr.trial_steps[n * p.trials + trial] = step;
        tr.trial_reward[n * p.trials + trial] = tw;
      }
      const int adv = live ? 33 : 0;
      rd = (rd + adv) & (kRing - 1); avail -= adv;
      nsteps += live ? 1 : 0;
      treward = tw;
      trial += (live && fin) ? 1 : 0;
      fresh = fin;
      step = step + 1;
      s = s2;
      live = live && trial < p.trials;
    }
  }

  __syncwarp();
  if (mine) {
    for (int e = h; e < SA; e += 16) {
      p.Q[g0 + e] = Q[e];
      p.Mr[g0 + e] = Mr[e];
      p.Ms[g0 + e] = Mx[e] & 0x7FFF;
      p.Mt[g0 + e] = Mx[e] >> 15;
    }
    if (h == 0) {
      p.stream.draw_count[n] = (int64_t)(gblk * 2) - (int64_t)avail;
      tr.n_steps[n] += nsteps;
      tr.n_replay[n] += (int64_t)nsteps * 32;
    }
  }
}

template <int A>
int launch(const CobelDynaQParams& p, cudaStream_t st) {
  const int S = p.world.n_states, K = p.world.n_starts;
  const WorldSmem wo(S, A, K);
  const bool plain = !p.action_mask && !p.world.tp_off && !p.trace.step_sa && !p.trace.step_td && !p.trace.replay_idx &&
                     !p.trace.replay_len &&
                     p.policy.kind == COBEL_POLICY_EPS_GREEDY && p.learn && !p.no_replay && !p.episodic_replay &&
                     p.batch == 32 && !p.stream.user_stream;
  const AgentSmem ao(S, A, plain);
  const size_t sm = (size_t)wo.bytes + (size_t)kWarpsPerCta * ao.bytes;
  const unsigned grid = (unsigned)((p.n_agents + kWarpsPerCta - 1) / kWarpsPerCta);
  if (sm > kMaxSmem) {
    // the tables do not fit: they stay in HBM / L2, only the dependency masks of the replay are staged
    const AgentSmem go(S, A, false, false);
    int warps = kWarpsPerCta;
    while (warps > 1 && (size_t)warps * go.bytes > kMaxSmem) warps >>= 1;
    const size_t smg = (size_t)warps * go.bytes;
    COBEL_REQUIRE(smg <= kMaxSmem, COBEL_EUNSUPPORTED,
                  "Dyna-Q: the replay's dependency masks of %d states do not fit in shared memory (%zu bytes)", S, smg);
    return launch_kernel(dynaq_warp_kernel<A, false, true>, (unsigned)((p.n_agents + warps - 1) / warps), warps * 32, smg, st, p);
  }
  if constexpr (A <= 4) {
    // The production case from two waves of the warp-per-agent kernel on: two agents per warp.  It pays once the
    // machine is full either way: with fewer agents the halved number of warps costs more issue rate than the shared
    // instructions save.  B200 at 1000 W, both kernels with the speculative replay pass: 4096 agents 2.30e9 against
    // 2.73e9 agent-steps/s, 16384 agents 3.58e9 against 3.40e9 (before that pass: 1.39e9 / 1.58e9 and 2.26e9 / 2.05e9).
    const PairSmem po(S, A);
    const size_t smp = (size_t)wo.bytes + (size_t)kPairWarps * 2 * po.bytes;
    static const int n_sm = [] { int d = 0, v = 148; if (cudaGetDevice(&d) == cudaSuccess) cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, d); return v; }();
    if (plain && p.n_agents >= (int64_t)2 * 7 * kWarpsPerCta * n_sm && smp <= kMaxSmem && S <= 0x7FFF) {
      const int64_t per_cta = kPairWarps * 2;
      return launch_kernel(dynaq_pair_kernel<A>, (unsigned)((p.n_agents + per_cta - 1) / per_cta), kPairWarps * 32, smp, st, p);
    }
    // the row summaries (9 bytes per state and agent) where they fit; otherwise the PLAIN kernel without them, so
    // that the largest world on chip stays the same
    const size_t sms = (size_t)wo.bytes + (size_t)kWarpsPerCta * AgentSmem(S, A, true, true, true).bytes;
    if (plain && sms <= kMaxSmem)
      return launch_kernel(dynaq_warp_kernel<A, true, false, true>, grid, kWarpsPerCta * 32, sms, st, p);
  }
  return launch_kernel(plain ? dynaq_warp_kernel<A, true> : dynaq_warp_kernel<A, false>, grid, kWarpsPerCta * 32, sm,
                       st, p);
}

}  // namespace

extern "C" int cobel_dynaq_run(const CobelDynaQParams* pp, void* stream) {
  COBEL_REQUIRE(pp != nullptr, COBEL_EINVAL, "null params");
  const CobelDynaQParams& p = *pp;
  int rc = cobel_validate_common(p.n_agents, p.world, p.stream, p.policy, p.trace, p.trials, p.steps);
  if (rc) return rc;
  COBEL_REQUIRE(p.Q && p.Mr && p.Ms && p.Mt && p.lr && p.gamma && p.mem_lr, COBEL_EINVAL, "agent tables missing");
  COBEL_REQUIRE(p.batch >= 0, COBEL_EINVAL, "batch must be >= 0");
  if (p.trials == 0) return COBEL_OK;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  COBEL_DISPATCH_A(p.world.n_actions, return launch<A>(p, st));
}
