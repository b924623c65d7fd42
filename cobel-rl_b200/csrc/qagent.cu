// qagent.cu -- K2: QAgent.train()/test() (tabular Q-learning with an append-only experience log)
// for N independent agents in one launch, on Gridworld or Topology-graph tables.
//
// Reference: agent/q.py:160-354.  Per step: select on Q[obs], environment step, append the
// experience to the log M, online TD update, then `batch` uniform draws over the WHOLE log
// (rng.choice(len(M), batch), q.py:353 -- the log already contains the current step) applied in
// order.  Q rows are keyed by observation (q.py:152-158): `obs_key[node]` is the row of a node
// (identity for gridworld states; index of the first node with the same pose for Topology).
//
// Mapping: one warp per agent, Q in shared memory, the log in HBM ([N, log_cap] 16-byte
// records: one LDG.128 per replayed experience, gathered one per lane); replayed updates run
// level-parallel exactly like Dyna-Q's (warp_agent.cuh).
#include "warp_agent.cuh"

namespace {

constexpr int kWarpsPerCta = 4;

struct __align__(16) LogRecord {
  double reward;
  uint16_t state, next_state;   // observation keys
  uint8_t action, nonterminal;
  uint16_t pad;
};
static_assert(sizeof(LogRecord) == 16, "log record must be 16 bytes");

struct QSmem {
  int q, wm, rm, ptab, draws, bytes;
  // table = false: Q stays in HBM (key spaces whose table does not fit), only the dependency masks are on chip
  __host__ __device__ QSmem(int NK, int A, bool table = true) {
    q = 0; wm = q + (table ? NK * A * 8 : 0); rm = wm + NK * 4; ptab = (rm + NK * 4 + 15) & ~15;
    draws = ptab + kEpsTabDoubles * 8;   // tie-pattern CDF table and stream window of the PLAIN kernel (warp_agent.cuh)
    bytes = draws + kSmemDraws * 8;
  }
};
struct QWorldSmem {
  int rew, succ, starts, key, term, bytes;
  __host__ __device__ QWorldSmem(int S, int A, int K) {
    rew = 0; succ = rew + S * 8; starts = succ + S * A * 4; key = starts + K * 4; term = key + S * 4;
    bytes = (term + S + 15) & ~15;
  }
};

// PLAIN = no optional trace buffers, deterministic world (see dynaq.cu)
// HBM = Q and the environment's tables stay in HBM / L2 (see dynaq.cu): only the dependency masks are on chip
template <int A, bool PLAIN, bool HBM = false>
__global__ void __launch_bounds__(kWarpsPerCta * 32, HBM ? 1 : 7) q_warp_kernel(const __grid_constant__ CobelQParams p) {
  static_assert(!(PLAIN && HBM), "the HBM path is the generic kernel");
  extern __shared__ __align__(16) unsigned char smem[];
  const int S = p.world.n_states, K = p.world.n_starts, NK = p.n_keys;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const QWorldSmem wo(HBM ? 0 : S, A, HBM ? 0 : K);
  const QSmem ao(NK, A, !HBM);
  double* rew_s = reinterpret_cast<double*>(smem + wo.rew);
  int32_t* succ_s = reinterpret_cast<int32_t*>(smem + wo.succ);
  int32_t* starts_s = reinterpret_cast<int32_t*>(smem + wo.starts);
  int32_t* key_s = reinterpret_cast<int32_t*>(smem + wo.key);
  uint8_t* term_s = smem + wo.term;
  if constexpr (!HBM) {
    for (int e = threadIdx.x; e < S * A; e += blockDim.x) succ_s[e] = p.world.succ[e];
    for (int e = threadIdx.x; e < S; e += blockDim.x) {
      rew_s[e] = p.world.reward[e]; term_s[e] = p.world.terminal[e];
      key_s[e] = p.obs_key ? p.obs_key[e] : e;
    }
    for (int e = threadIdx.x; e < K; e += blockDim.x) starts_s[e] = p.world.starts[e];
    __syncthreads();
  }
  auto w_succ = [&](int sa) -> int { if constexpr (HBM) return __ldg(p.world.succ + sa); else return succ_s[sa]; };
  auto w_rew = [&](int x) -> double { if constexpr (HBM) return __ldg(p.world.reward + x); else return rew_s[x]; };
  auto w_term = [&](int x) -> int { if constexpr (HBM) return __ldg(p.world.terminal + x); else return term_s[x]; };
  auto w_start = [&](int k) -> int { if constexpr (HBM) return __ldg(p.world.starts + k); else return starts_s[k]; };
  auto w_key = [&](int x) -> int { if constexpr (HBM) return p.obs_key ? __ldg(p.obs_key + x) : x; else return key_s[x]; };

  const int64_t n = (int64_t)blockIdx.x * blockDim.x / 32 + warp;
  if (n >= p.n_agents) return;
  unsigned char* blk = smem + wo.bytes + (size_t)warp * ao.bytes;
  const size_t g0 = (size_t)n * NK * A;
  double* Q = HBM ? p.Q + g0 : reinterpret_cast<double*>(blk + ao.q);
  uint32_t* wm = reinterpret_cast<uint32_t*>(blk + ao.wm);
  uint32_t* rm = reinterpret_cast<uint32_t*>(blk + ao.rm);
  if constexpr (!HBM)
    for (int e = lane; e < NK * A; e += 32) Q[e] = p.Q[g0 + e];
  for (int e = lane; e < NK; e += 32) { wm[e] = 0; rm[e] = 0; }
  __syncwarp();

  typename WindowFor<PLAIN>::type win; win.init(p.stream, n, (uint64_t)p.stream.draw_count[n]);
  win.attach(reinterpret_cast<double*>(blk + ao.draws));
  const double lr = p.lr[n], gamma = p.gamma[n];
  PolicyTab pt; pt.init(p.policy.kind, p.policy.param[n], lane);
  constexpr bool kEpsTab = PLAIN && A <= 4;
  double* ptab = reinterpret_cast<double*>(blk + ao.ptab);
  if constexpr (kEpsTab) eps_cdf_table_init<A>(ptab, pt, lane);
  const int B = PLAIN ? 32 : p.batch;
  const bool learn = PLAIN || p.learn != 0;
  LogRecord* log = reinterpret_cast<LogRecord*>(p.log) + (size_t)n * p.log_cap;
  int64_t len = learn ? p.log_len[n] : 0;
  const CobelTrace& tr = p.trace;
  int64_t nsteps = 0, nrep = 0, ncalls = 0;
  int flags = 0;

  for (int trial = 0; trial < p.trials; ++trial) {
    win.ensure(3 + (learn && B <= 32 ? B : 0), lane);
    int s = w_start(draw_integer(win.next(), K));                 // interface reset: one draw
    double treward = 0.0;
    int step = 0;
    for (;; ++step) {
      win.ensure(2 + (learn && B <= 32 ? B : 0), lane);
      const int ks = w_key(s);
      double row[A];
      load_row<A>(Q + ks * A, row);
      int a;
      if constexpr (kEpsTab) a = select_action_eps_tab<A>(row, ptab, win.next(), lane);
      else a = select_action_warp<A, PLAIN ? COBEL_POLICY_EPS_GREEDY : -1>(row, (1u << A) - 1u, pt, win.next(), lane);
      const int s2 = (!PLAIN && p.world.tp_off) ? stochastic_successor(p.world, s * A + a, win.next()) : w_succ(s * A + a);
      const double r = w_rew(s2);
      const int end = w_term(s2);
      const int nt = 1 - end;
      const int ks2 = w_key(s2);
      if (!PLAIN && tr.step_sa && lane == 0) {
        if (nsteps < tr.step_cap) { tr.step_sa[n * tr.step_cap + nsteps] = s * A + a; if (tr.step_next) tr.step_next[n * tr.step_cap + nsteps] = s2; }
        else flags |= COBEL_FLAG_TRACE_OVERFLOW;
      }
      ++nsteps;
      if (learn) {
        // q.py:213-214: append, then the online update (q.py:297-322)
        double row2[A];
        load_row<A>(Q + ks2 * A, row2);
        const double q = Q[ks * A + a];
        const double g = nt ? gamma : 0.0;
        double td = xadd(r, xmul(g, row_max<A>(row2)));
        td = xsub(td, q);
        const double qn = xadd(q, xmul(lr, td));
        if (!PLAIN && tr.step_td && lane == 0) {     // the step's slot of step_sa (nsteps already counts it)
          if (nsteps <= tr.step_cap) tr.step_td[n * tr.step_cap + nsteps - 1] = td;
          else flags |= COBEL_FLAG_TRACE_OVERFLOW;
        }
        const bool room = len < p.log_cap;
        __syncwarp();
        if (lane == 0) {
          if (room) {
            LogRecord rec{r, (uint16_t)ks, (uint16_t)ks2, (uint8_t)a, (uint8_t)nt, 0};
            log[len] = rec;
          }
          Q[ks * A + a] = qn;
        }
        if (room) ++len; else flags |= COBEL_FLAG_LOG_OVERFLOW;
        __syncwarp();
        // q.py:344-354: `batch` uniform draws over the log, applied in order
        for (int b0 = 0; b0 < B; b0 += 32) {
          const int nb = B - b0 < 32 ? B - b0 : 32;
          win.ensure(nb, lane);
          const bool active = lane < nb;
          const double u = win.peek(active ? lane : 0);
          win.advance(nb);
          int es = 0, ea = 0, es2 = 0, ent = 0;
          double er = 0.0;
          if (active) {
            const int i = draw_integer(u, (int)len);
            const LogRecord rec = log[i];
            es = rec.state; ea = rec.action; es2 = rec.next_state; ent = rec.nonterminal; er = rec.reward;
            if (!PLAIN && tr.replay_idx) {
              if (nrep + lane < tr.replay_cap) tr.replay_idx[n * tr.replay_cap + nrep + lane] = i;
              else flags |= COBEL_FLAG_TRACE_OVERFLOW;
            }
          }
          td_batch_level_parallel<A>(Q, wm, rm, NK, lane, active, es, ea, er, es2, ent, lr, gamma);
          nrep += nb;
        }
        if (!PLAIN && tr.replay_len && lane == 0) {  // one replay call per step, also for batch 0 (q.py:216)
          if (ncalls < tr.replay_calls_cap) tr.replay_len[n * tr.replay_calls_cap + ncalls] = B;
          else flags |= COBEL_FLAG_TRACE_OVERFLOW;
        }
        ++ncalls;
      }
      s = s2;
      treward = xadd(treward, r);
      if (end || step + 1 == p.steps) break;
    }
    if (lane == 0) {
      tr.trial_steps[n * p.trials + trial] = step;
      tr.trial_reward[n * p.trials + trial] = treward;
    }
  }

  __syncwarp();
  if (learn && !HBM)
    for (int e = lane; e < NK * A; e += 32) p.Q[g0 + e] = Q[e];
  flags = __reduce_or_sync(kFull, flags);
  if (lane == 0) {
    p.stream.draw_count[n] = (int64_t)win.position();
    if (learn) p.log_len[n] = len;
    tr.n_steps[n] += nsteps;
    tr.n_replay[n] += nrep;
    if (tr.flags && flags) tr.flags[n] |= flags;
  }
}

template <int A>
int launch(const CobelQParams& p, cudaStream_t st) {
  const QWorldSmem wo(p.world.n_states, A, p.world.n_starts);
  const QSmem ao(p.n_keys, A);
  const size_t sm = (size_t)wo.bytes + (size_t)kWarpsPerCta * ao.bytes;
  if (sm > kMaxSmem) {
    // the tables do not fit: Q stays in HBM / L2, only the dependency masks of the replay are staged
    const QSmem go(p.n_keys, A, false);
    int warps = kWarpsPerCta;
    while (warps > 1 && (size_t)warps * go.bytes > kMaxSmem) warps >>= 1;
    const size_t smg = (size_t)warps * go.bytes;
    COBEL_REQUIRE(smg <= kMaxSmem, COBEL_EUNSUPPORTED,
                  "QAgent: the replay's dependency masks of %d keys do not fit in shared memory (%zu bytes)", p.n_keys, smg);
    return launch_kernel(q_warp_kernel<A, false, true>, (unsigned)((p.n_agents + warps - 1) / warps), warps * 32, smg, st, p);
  }
  const bool plain = !p.world.tp_off && !p.trace.step_sa && !p.trace.step_td && !p.trace.replay_idx && !p.trace.replay_len &&
                     p.policy.kind == COBEL_POLICY_EPS_GREEDY && p.learn && p.batch == 32 && !p.stream.user_stream;
  return launch_kernel(plain ? q_warp_kernel<A, true> : q_warp_kernel<A, false>,
                       (unsigned)((p.n_agents + kWarpsPerCta - 1) / kWarpsPerCta), kWarpsPerCta * 32, sm, st, p);
}

}  // namespace

extern "C" int cobel_q_run(const CobelQParams* pp, void* stream) {
  COBEL_REQUIRE(pp != nullptr, COBEL_EINVAL, "null params");
  const CobelQParams& p = *pp;
  int rc = cobel_validate_common(p.n_agents, p.world, p.stream, p.policy, p.trace, p.trials, p.steps);
  if (rc) return rc;
  COBEL_REQUIRE(p.Q && p.lr && p.gamma, COBEL_EINVAL, "agent tables missing");
  COBEL_REQUIRE(p.n_keys > 0 && p.n_keys <= 65535, COBEL_EINVAL, "n_keys must be in 1..65535");
  COBEL_REQUIRE(p.batch >= 0, COBEL_EINVAL, "batch must be >= 0");
  if (p.trials == 0) return COBEL_OK;                  // a zero-trial session is a no-op (no log needed)
  COBEL_REQUIRE(!p.learn || (p.log && p.log_len && p.log_cap > 0), COBEL_EINVAL, "experience log missing");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  COBEL_DISPATCH_A(p.world.n_actions, return launch<A>(p, st));
}
