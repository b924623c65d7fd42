// ops.cu -- the stand-alone methods of the class API, one call = one method of the reference for all N agents:
// Interface.reset/step, Policy.get_action_probs/select_action, Memory.store/retrieve_batch, Agent.update_q/replay,
// SR.update/retrieve_q, PMAMemory.compute_gain_batch/compute_need.  They serve callers that drive the loop
// themselves (env.step -> policy.select_action -> M.store -> agent.update_q -> agent.replay, agent/dyna_q.py:176-203)
// instead of the fused train(); same arithmetic (thread_agent.cuh), same stream contract (one uniform stream per
// agent, consumed in program order).  One thread per agent: a method touches a handful of table entries.
// PMAMemory.replay and SFMAMemory.replay are phases of the fused kernels (pma.cu, sfma.cu).
#include "thread_agent.cuh"

namespace {

constexpr int kT = 128;
inline unsigned grid_for(int64_t n) { return (unsigned)((n + kT - 1) / kT); }

// ---- environment: interface/gridworld.py:92-145, interface/topology.py:126-172 --------------------------------
__global__ void env_reset_kernel(CobelWorld w, CobelStream s, int64_t n_agents, int32_t* state) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_agents) return;
  Rng rng; rng.init(s, n);
  state[n] = __ldg(w.starts + draw_integer(rng.next(), w.n_starts));
  s.draw_count[n] = (int64_t)rng.k;
}

__global__ void env_step_kernel(CobelWorld w, CobelStream s, int64_t n_agents, int32_t* state, const int32_t* action,
                                double* reward, uint8_t* end_trial) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_agents) return;
  const int sa = state[n] * w.n_actions + action[n];
  int s2;
  if (w.tp_off) {                                     // gridworld.py:118-123: one categorical draw over sas[s, a, :]
    Rng rng; rng.init(s, n);
    s2 = stochastic_successor_t(w, sa, rng.next());
    s.draw_count[n] = (int64_t)rng.k;
  } else {
    s2 = __ldg(w.succ + sa);
  }
  state[n] = s2;
  reward[n] = __ldg(w.reward + s2);
  end_trial[n] = __ldg(w.terminal + s2);
}

// ---- policies: policy/greedy.py:40-147, policy/softmax.py:40-88 ---------------------------------------------------
COBEL_DEV uint32_t row_mask_bits(const uint8_t* mask, int64_t row, int A) {
  uint32_t mb = (1u << A) - 1u;
  if (mask) {
    mb = 0;
    for (int a = 0; a < A; ++a) mb |= (mask[row * A + a] ? 1u : 0u) << a;
  }
  return mb;
}

template <int A>
__global__ void policy_probs_kernel(CobelPolicy pol, int64_t n_rows, int64_t rows_per_agent, const double* values,
                                    const uint8_t* mask, double* probs) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  double v[A], p[A];
#pragma unroll
  for (int a = 0; a < A; ++a) v[a] = values[r * A + a];
  action_probs_thread<A>(v, row_mask_bits(mask, r, A), pol.kind, pol.param[r / rows_per_agent], p);
#pragma unroll
  for (int a = 0; a < A; ++a) probs[r * A + a] = p[a];
}

template <int A>
__global__ void policy_select_kernel(CobelPolicy pol, CobelStream s, int64_t n_agents, const double* values,
                                     const uint8_t* mask, int32_t* action) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_agents) return;
  double v[A];
#pragma unroll
  for (int a = 0; a < A; ++a) v[a] = values[n * A + a];
  Rng rng; rng.init(s, n);
  action[n] = select_action_thread<A>(v, row_mask_bits(mask, n, A), pol.kind, pol.param[n], rng.next());
  s.draw_count[n] = (int64_t)rng.k;
}

// ---- experiences ------------------------------------------------------------------------------------------------------
struct Exp { int s, a, s2, nt; double r; };
COBEL_DEV Exp exp_at(const CobelExperiences& e, int64_t n, int b) {
  const int64_t i = n * e.batch + b;
  return Exp{e.state[i], e.action[i], e.next_state[i], e.terminal[i] ? 1 : 0, e.reward[i]};
}
COBEL_DEV void exp_put(const CobelExperiences& e, int64_t n, int b, int s, int a, double r, int s2, int nt) {
  const int64_t i = n * e.batch + b;
  e.state[i] = s; e.action[i] = a; e.reward[i] = r; e.next_state[i] = s2; e.terminal[i] = nt;
}

// ---- Dyna-Q: memory/dyna_q.py:77-157, agent/dyna_q.py:275-330 ----------------------------------------------------
template <int A>
__global__ void dynaq_op_kernel(CobelDynaQParams p, int op, CobelExperiences e) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.n_agents) return;
  const int S = p.world.n_states;
  const size_t g0 = (size_t)n * S * A;
  double* Q = p.Q + g0; double* Mr = p.Mr + g0; int32_t* Ms = p.Ms + g0; int32_t* Mt = p.Mt + g0;
  constexpr uint32_t kAll = (1u << A) - 1u;        // DynaQ.update_q takes the max over all actions of s'
  if (op == COBEL_OP_STORE) {                       // DynaQMemory.store
    const Exp x = exp_at(e, n, 0);
    const double m0 = Mr[x.s * A + x.a];
    Mr[x.s * A + x.a] = xadd(m0, xmul(p.mem_lr[n], xsub(x.r, m0)));
    Ms[x.s * A + x.a] = x.s2;
    Mt[x.s * A + x.a] = x.nt;
  } else if (op == COBEL_OP_UPDATE_Q) {             // DynaQ.update_q for every experience of the batch, in order
    for (int b = 0; b < e.batch; ++b) {
      const Exp x = exp_at(e, n, b);
      const double td = td_update_thread<A>(Q, x.s, x.a, x.r, x.s2, x.nt, p.lr[n], p.gamma[n], kAll);
      if (e.td) e.td[n * e.batch + b] = td;
    }
  } else {                                          // retrieve_batch [+ update_q]: batch uniform draws over S*A, C order
    Rng rng; rng.init(p.stream, n);
    for (int b = 0; b < e.batch; ++b) {
      const int i = draw_integer(rng.next(), S * A);
      const int s = i / A, a = i - s * A;
      exp_put(e, n, b, s, a, Mr[i], Ms[i], Mt[i]);
    }
    p.stream.draw_count[n] = (int64_t)rng.k;
    if (op == COBEL_OP_REPLAY) {                    // DynaQ.replay: the whole batch is drawn first, then applied in order
      for (int b = 0; b < e.batch; ++b) {
        const Exp x = exp_at(e, n, b);
        const double td = td_update_thread<A>(Q, x.s, x.a, x.r, x.s2, x.nt, p.lr[n], p.gamma[n], kAll);
        if (e.td) e.td[n * e.batch + b] = td;
      }
      if (p.trace.n_replay) p.trace.n_replay[n] += e.batch;
    }
  }
}

// ---- QAgent: agent/q.py:205-215 (append), 297-354 ------------------------------------------------------------------
struct __align__(16) LogRecord {
  double reward;
  uint16_t state, next_state;   // observation keys
  uint8_t action, nonterminal;
  uint16_t pad;
};

template <int A>
__global__ void q_op_kernel(CobelQParams p, int op, CobelExperiences e) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.n_agents) return;
  double* Q = p.Q + (size_t)n * p.n_keys * A;
  LogRecord* log = reinterpret_cast<LogRecord*>(p.log) + (size_t)n * p.log_cap;
  constexpr uint32_t kAll = (1u << A) - 1u;
  auto key = [&](int s) -> int { return p.obs_key ? p.obs_key[s] : s; };
  if (op == COBEL_OP_STORE) {                       // self.M.append(experience)
    const Exp x = exp_at(e, n, 0);
    const int64_t len = p.log_len[n];
    if (len < p.log_cap) {
      log[len] = LogRecord{x.r, (uint16_t)key(x.s), (uint16_t)key(x.s2), (uint8_t)x.a, (uint8_t)x.nt, 0};
      p.log_len[n] = len + 1;
    } else if (p.trace.flags) {
      p.trace.flags[n] |= COBEL_FLAG_LOG_OVERFLOW;
    }
  } else if (op == COBEL_OP_UPDATE_Q) {
    for (int b = 0; b < e.batch; ++b) {
      const Exp x = exp_at(e, n, b);
      const double td = td_update_thread<A>(Q, key(x.s), x.a, x.r, key(x.s2), x.nt, p.lr[n], p.gamma[n], kAll);
      if (e.td) e.td[n * e.batch + b] = td;
    }
  } else if (op == COBEL_OP_REPLAY) {               // for i in rng.choice(len(M), batch): update_q(M[i])
    Rng rng; rng.init(p.stream, n);
    const int len = (int)p.log_len[n];
    for (int b = 0; b < e.batch; ++b) {
      const int i = draw_integer(rng.next(), len);
      if (e.state) e.state[n * e.batch + b] = i;     // the log index of the replayed experience
      if (p.trace.replay_idx) p.trace.replay_idx[n * p.trace.replay_cap + b] = i;
    }
    for (int b = 0; b < e.batch; ++b) {
      const LogRecord x = log[e.state[n * e.batch + b]];
      td_update_thread<A>(Q, x.state, x.action, x.reward, x.next_state, x.nonterminal, p.lr[n], p.gamma[n], kAll);
    }
    p.stream.draw_count[n] = (int64_t)rng.k;
    if (p.trace.n_replay) p.trace.n_replay[n] += e.batch;
  }
}

// ---- SR agent: agent/sr.py:255-308 -----------------------------------------------------------------------------------
// NumPy's pairwise sum of x[i] * y[i], i < n (np.sum over one contiguous row): blocks of <= 128 elements with 8
// accumulators, recursive halving above (SURVEY.md Appendix A.3)
__device__ double pairwise_dot(const double* x, const double* y, int n) {
  if (n < 8) {
    double r = 0.0;
    for (int i = 0; i < n; ++i) r = xadd(r, xmul(x[i], y[i]));
    return r;
  }
  if (n <= 128) {
    double r[8];
    for (int j = 0; j < 8; ++j) r[j] = xmul(x[j], y[j]);
    int i = 8;
    for (; i < n - (n % 8); i += 8)
      for (int j = 0; j < 8; ++j) r[j] = xadd(r[j], xmul(x[i + j], y[i + j]));
    double res = xadd(xadd(xadd(r[0], r[1]), xadd(r[2], r[3])), xadd(xadd(r[4], r[5]), xadd(r[6], r[7])));
    for (; i < n; ++i) res = xadd(res, xmul(x[i], y[i]));
    return res;
  }
  int n2 = n / 2;
  n2 -= n2 % 8;
  return xadd(pairwise_dot(x, y, n2), pairwise_dot(x + n2, y + n2, n - n2));
}

template <int A>
__global__ void sr_op_kernel(CobelSRParams p, int op, CobelExperiences e, const int32_t* state, double* q_out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.n_agents) return;
  const int S = p.world.n_states;
  double* SR = p.SR + (size_t)n * S * S;
  double* rew = p.rewards + (size_t)n * S;
  int32_t* model = p.model + (size_t)n * S * A;
  if (op == COBEL_OP_STORE) {                       // SR.update(experience), agent/sr.py:255-286
    const Exp x = exp_at(e, n, 0);
    const double lr = p.lr[n], gamma = p.gamma[n];
    const double tdr = xsub(x.r, rew[x.s2]);
    rew[x.s2] = xadd(rew[x.s2], xmul(tdr, lr));
    model[x.s * A + x.a] = x.s2;
    double* row = SR + (size_t)x.s * S;
    const double* nxt = SR + (size_t)x.s2 * S;
    for (int j = 0; j < S; ++j) {
      // td = e_s + gamma * (SR[s'] if terminal > 0 else e_s') - SR[s]; a row is updated from its own old values and
      // from SR[s'] -- for s' == s the old value of the same element, read before it is written
      const double boot = x.nt ? nxt[j] : (j == x.s2 ? 1.0 : 0.0);
      double td = xadd(j == x.s ? 1.0 : 0.0, xmul(gamma, boot));
      td = xsub(td, row[j]);
      row[j] = xadd(row[j], xmul(lr, td));
    }
  } else {                                          // SR.retrieve_q(state), agent/sr.py:288-308
    const int s = state[n];
    for (int a = 0; a < A; ++a) q_out[n * A + a] = pairwise_dot(SR + (size_t)model[s * A + a] * S, rew, S);
  }
}

// ---- SFMA: memory/sfma.py:195-236 (store), agent/sfma.py:423-458 (update_q) -----------------------------------------
template <int A>
__global__ void sfma_op_kernel(CobelSFMAParams p, int op, CobelExperiences e) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.n_agents) return;
  const int S = p.world.n_states, N = S * A;
  const size_t g0 = (size_t)n * N;
  double* Q = p.Q + g0; double* Mr = p.Mr + g0; int32_t* Ms = p.Ms + g0; int32_t* Mt = p.Mt + g0;
  double* C = p.C + g0; double* T = p.T + g0;
  const uint8_t* amask = p.action_mask ? p.action_mask + n * p.mask_agent_stride : nullptr;
  if (op == COBEL_OP_STORE) {
    const Exp x = exp_at(e, n, 0);
    const int i = x.a * S + x.s;
    const double m0 = Mr[x.s * A + x.a];
    Mr[x.s * A + x.a] = xadd(m0, xmul(p.mem_lr[n], xsub(x.r, m0)));
    Ms[x.s * A + x.a] = x.s2;
    Mt[x.s * A + x.a] = x.nt;
    if (p.decay_strength != 1.0)
      for (int j = 0; j < N; ++j) C[j] = xmul(C[j], p.decay_strength);
    C[i] = xadd(C[i], p.c_step);
    for (int j = 0; j < N; ++j) T[j] = xmul(T[j], p.decay_recency);
    T[i] = 1.0;
    if (p.mod_flags & COBEL_SFMA_MOD_REWARD_LOCAL) C[i] = xadd(C[i], xmul(x.r, p.reward_modulation));
    if (p.mod_flags & COBEL_SFMA_MOD_REWARD) {
      const double* Ds = p.D + (size_t)x.s * S;
      for (int j = 0; j < N; ++j) C[j] = xadd(C[j], xmul(xmul(x.r, Ds[j % S]), p.reward_modulation));
    }
    if (p.mod_flags & COBEL_SFMA_MOD_STATE)
      for (int a = 0; a < A; ++a) C[a * S + x.s] = xadd(C[a * S + x.s], 1.0);
  } else if (op == COBEL_OP_UPDATE_Q) {             // masked max over Q[s'], agent.td += |td|; no_update via p.learn == 0
    double tdacc = p.td_acc ? p.td_acc[n] : 0.0;
    for (int b = 0; b < e.batch; ++b) {
      const Exp x = exp_at(e, n, b);
      const double td = td_update_thread<A>(Q, x.s, x.a, x.r, x.s2, x.nt, p.lr[n], p.gamma[n], mask_bits<A>(amask, x.s2),
                                            p.learn != 0);
      if (e.td) e.td[n * e.batch + b] = td;
      tdacc = xadd(tdacc, fabs(td));
    }
    if (p.td_acc) p.td_acc[n] = tdacc;
  } else if (op == COBEL_OP_GATHER) {               // the experiences behind flat indices a*S + s (in e.state): fills e
    for (int b = 0; b < e.batch; ++b) {
      const int i = e.state[n * e.batch + b];
      if (i < 0) { exp_put(e, n, b, -1, -1, 0.0, -1, 0); continue; }
      const int a = i / S, s = i - a * S;
      exp_put(e, n, b, s, a, Mr[s * A + a], Ms[s * A + a], Mt[s * A + a]);
    }
  }
}

// ---- PMA: memory/pma.py:148-166 (store), agent/pma.py:319-353 (update_q), memory/pma.py:333-411 ----------------------
template <int A>
__global__ void pma_op_kernel(CobelPMAParams p, int op, CobelExperiences e, const int32_t* state, double* out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.n_agents) return;
  const int S = p.world.n_states, N = S * A;
  const size_t g0 = (size_t)n * N;
  double* Q = p.Q + g0; double* Mr = p.Mr + g0; int32_t* Ms = p.Ms + g0; int32_t* Mt = p.Mt + g0;
  if (op == COBEL_OP_STORE) {                       // PMAMemory.store: table entry + T[s] += lr_T (onehot(s') - T[s])
    const Exp x = exp_at(e, n, 0);
    const double m0 = Mr[x.s * A + x.a];
    Mr[x.s * A + x.a] = xadd(m0, xmul(p.mem_lr[n], xsub(x.r, m0)));
    Ms[x.s * A + x.a] = x.s2;
    Mt[x.s * A + x.a] = x.nt;
    double* Trow = p.T + ((size_t)n * S + x.s) * S;
    for (int j = 0; j < S; ++j) Trow[j] = xadd(Trow[j], xmul(p.lr_T, xsub(j == x.s2 ? 1.0 : 0.0, Trow[j])));
  } else if (op == COBEL_OP_UPDATE_Q) {             // PMA.update_q: the batch is ONE n-step update; pow_gamma_q = agent.gamma ** k
    const int nseq = e.batch;
    const double* powg = p.pow_gamma_q + n * p.pow_stride;
    const Exp last = exp_at(e, n, nseq - 1);
    double row[A];
    load_row_t<A>(Q + (size_t)last.s2 * A, row);
    const double fv = xmul(row_max<A>(row), last.nt ? 1.0 : 0.0);
    for (int j = 0; j < nseq; ++j) {
      double r = 0.0;
      bool ok = true;
      int f = 0;
      for (; f < nseq - j; ++f) {
        const Exp y = exp_at(e, n, j + f);
        if (y.nt == 0 && j != nseq - 1) { ok = false; break; }
        r = xadd(r, xmul(y.r, powg[f]));
      }
      if (!ok) break;
      const Exp x = exp_at(e, n, j);
      double td = xadd(r, xmul(fv, powg[nseq - j]));
      const double q = Q[x.s * A + x.a];
      td = xsub(td, q);
      Q[x.s * A + x.a] = xadd(q, xmul(p.lr[n], td));
    }
  } else if (op == COBEL_OP_NEED) {                 // compute_need(current_state): tile(SR[state]) or tile(stationary need)
    const int s = state[n];
    const double* src = s >= 0 ? p.SR + ((size_t)n * S + s) * S : p.need_scratch + (size_t)n * S;
    for (int i = 0; i < N; ++i) out[(size_t)n * N + i] = src[i % S];
  }
}

// compute_gain_batch (memory/pma.py:333-386): one thread per (agent, one-step backup)
template <int A>
__global__ void pma_gain_batch_kernel(CobelPMAParams p, double* out) {
  const int S = p.world.n_states, N = S * A;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= p.n_agents * N) return;
  const int64_t n = t / N;
  const int i = (int)(t - n * N), a = i / S, s = i - a * S;
  const size_t g0 = (size_t)n * N;
  const double* Q = p.Q + g0;
  const uint8_t* amask = p.action_mask ? p.action_mask + n * p.mask_agent_stride : nullptr;
  double q[A], qn[A], tr_[A], po[A], pn[A], tt[A];
  load_row_t<A>(Q + (size_t)s * A, q);
  load_row_t<A>(Q + (size_t)p.Ms[g0 + s * A + a] * A, tr_);
  const double boot = xmul(xmul(p.gamma_q[n], row_max<A>(tr_)), p.Mt[g0 + s * A + a] ? 1.0 : 0.0);
  const double qa = pick_reg<A>(q, a);
  const double upd = xadd(qa, xmul(p.lr_q[n], xsub(xadd(p.Mr[g0 + s * A + a], boot), qa)));
#pragma unroll
  for (int c = 0; c < A; ++c) qn[c] = c == a ? upd : q[c];
  const uint32_t mb = mask_bits<A>(amask, s);
  action_probs_thread<A>(q, mb, p.mem_policy.kind, p.mem_policy.param[n], po);
  action_probs_thread<A>(qn, mb, p.mem_policy.kind, p.mem_policy.param[n], pn);
  const double so = np_sum<A>(po), sn = np_sum<A>(pn);
#pragma unroll
  for (int c = 0; c < A; ++c) { po[c] = xdiv(po[c], so); pn[c] = xdiv(pn[c], sn); }
#pragma unroll
  for (int c = 0; c < A; ++c) tt[c] = xmul(pn[c], qn[c]);
  const double gnew = np_sum<A>(tt);
#pragma unroll
  for (int c = 0; c < A; ++c) tt[c] = xmul(po[c], qn[c]);
  const double g = xsub(gnew, np_sum<A>(tt));
  out[t] = g > p.min_gain ? g : p.min_gain;
}

bool exp_ok(const CobelExperiences* e, bool need_fields) {
  return e && e->batch > 0 && (!need_fields || (e->state && e->action && e->reward && e->next_state && e->terminal));
}

}  // namespace

extern "C" int cobel_env_reset(const CobelWorld* w, const CobelStream* s, int64_t n_agents, int32_t* state, void* stream) {
  COBEL_REQUIRE(w && s && s->draw_count && state && n_agents > 0 && w->starts && w->n_starts > 0, COBEL_EINVAL, "bad arguments to cobel_env_reset");
  env_reset_kernel<<<grid_for(n_agents), kT, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*w, *s, n_agents, state);
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}

extern "C" int cobel_env_step(const CobelWorld* w, const CobelStream* s, int64_t n_agents, int32_t* state, const int32_t* action,
                              double* reward, uint8_t* end_trial, void* stream) {
  COBEL_REQUIRE(w && s && state && action && reward && end_trial && n_agents > 0 && w->succ && w->reward && w->terminal,
                COBEL_EINVAL, "bad arguments to cobel_env_step");
  COBEL_REQUIRE(!w->tp_off || s->draw_count, COBEL_EINVAL, "a non-deterministic world needs the stream");
  env_step_kernel<<<grid_for(n_agents), kT, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*w, *s, n_agents, state, action, reward, end_trial);
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}

extern "C" int cobel_policy_probs(const CobelPolicy* pol, int64_t n_agents, int64_t rows_per_agent, int32_t n_actions,
                                  const double* values, const uint8_t* mask, double* probs, void* stream) {
  COBEL_REQUIRE(pol && pol->param && pol->kind >= 0 && pol->kind <= 2 && values && probs && n_agents > 0 && rows_per_agent > 0,
                COBEL_EINVAL, "bad arguments to cobel_policy_probs");
  const int64_t rows = n_agents * rows_per_agent;
  COBEL_DISPATCH_A(n_actions, (policy_probs_kernel<A><<<grid_for(rows), kT, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
                                   *pol, rows, rows_per_agent, values, mask, probs)));
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}

extern "C" int cobel_policy_select(const CobelPolicy* pol, const CobelStream* s, int64_t n_agents, int32_t n_actions,
                                   const double* values, const uint8_t* mask, int32_t* action, void* stream) {
  COBEL_REQUIRE(pol && pol->param && pol->kind >= 0 && pol->kind <= 2 && s && s->draw_count && values && action && n_agents > 0,
                COBEL_EINVAL, "bad arguments to cobel_policy_select");
  COBEL_DISPATCH_A(n_actions, (policy_select_kernel<A><<<grid_for(n_agents), kT, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
                                   *pol, *s, n_agents, values, mask, action)));
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}

extern "C" int cobel_dynaq_op(const CobelDynaQParams* p, int op, const CobelExperiences* e, void* stream) {
  COBEL_REQUIRE(op == COBEL_OP_STORE || op == COBEL_OP_UPDATE_Q || op == COBEL_OP_RETRIEVE_BATCH || op == COBEL_OP_REPLAY,
                COBEL_EINVAL, "cobel_dynaq_op: unknown op %d", op);
  COBEL_REQUIRE(p && p->n_agents > 0 && p->world.n_states > 0, COBEL_EINVAL, "null / empty params");
  COBEL_REQUIRE(op == COBEL_OP_UPDATE_Q || (p->Mr && p->Ms && p->Mt), COBEL_EINVAL, "memory tables missing");
  COBEL_REQUIRE(op != COBEL_OP_STORE || p->mem_lr, COBEL_EINVAL, "mem_lr missing");
  COBEL_REQUIRE((op != COBEL_OP_UPDATE_Q && op != COBEL_OP_REPLAY) || (p->Q && p->lr && p->gamma), COBEL_EINVAL, "Q / lr / gamma missing");
  COBEL_REQUIRE(exp_ok(e, true), COBEL_EINVAL, "experience batch missing");
  COBEL_REQUIRE((op != COBEL_OP_RETRIEVE_BATCH && op != COBEL_OP_REPLAY) || p->stream.draw_count, COBEL_EINVAL, "stream missing");
  COBEL_DISPATCH_A(p->world.n_actions, (dynaq_op_kernel<A><<<grid_for(p->n_agents), kT, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*p, op, *e)));
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}

extern "C" int cobel_q_op(const CobelQParams* p, int op, const CobelExperiences* e, void* stream) {
  COBEL_REQUIRE(p && p->n_agents > 0 && p->Q && p->lr && p->gamma && p->log_len, COBEL_EINVAL, "agent tables missing");
  COBEL_REQUIRE(op == COBEL_OP_STORE || op == COBEL_OP_UPDATE_Q || op == COBEL_OP_REPLAY, COBEL_EINVAL, "cobel_q_op: unknown op %d", op);
  COBEL_REQUIRE(exp_ok(e, op != COBEL_OP_REPLAY) && (op != COBEL_OP_REPLAY || e->state), COBEL_EINVAL, "experience batch missing");
  COBEL_REQUIRE(op == COBEL_OP_UPDATE_Q || p->log, COBEL_EINVAL, "experience log missing");
  COBEL_REQUIRE(p->world.n_states <= 65535, COBEL_EUNSUPPORTED, "QAgent log records hold 16-bit observation keys");
  COBEL_DISPATCH_A(p->world.n_actions, (q_op_kernel<A><<<grid_for(p->n_agents), kT, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*p, op, *e)));
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}

extern "C" int cobel_sr_op(const CobelSRParams* p, int op, const CobelExperiences* e, const int32_t* state, double* q_out, void* stream) {
  COBEL_REQUIRE(p && p->n_agents > 0 && p->SR && p->rewards && p->model && p->lr && p->gamma, COBEL_EINVAL, "agent tables missing");
  COBEL_REQUIRE((op == COBEL_OP_STORE && exp_ok(e, true)) || (op == COBEL_OP_RETRIEVE_Q && state && q_out), COBEL_EINVAL,
                "cobel_sr_op: op must be COBEL_OP_STORE (SR.update, with an experience) or COBEL_OP_RETRIEVE_Q (with state and q_out)");
  CobelExperiences none{};
  COBEL_DISPATCH_A(p->world.n_actions, (sr_op_kernel<A><<<grid_for(p->n_agents), kT, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
                                            *p, op, e ? *e : none, state, q_out)));
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}

extern "C" int cobel_sfma_op(const CobelSFMAParams* p, int op, const CobelExperiences* e, void* stream) {
  COBEL_REQUIRE(op == COBEL_OP_STORE || op == COBEL_OP_UPDATE_Q || op == COBEL_OP_GATHER, COBEL_EINVAL, "cobel_sfma_op: unknown op %d", op);
  COBEL_REQUIRE(p && p->n_agents > 0 && p->world.n_states > 0, COBEL_EINVAL, "null / empty params");
  COBEL_REQUIRE(op == COBEL_OP_UPDATE_Q || (p->Mr && p->Ms && p->Mt), COBEL_EINVAL, "memory tables missing");
  COBEL_REQUIRE(op != COBEL_OP_STORE || (p->C && p->T && p->mem_lr), COBEL_EINVAL, "C / T / mem_lr missing");
  COBEL_REQUIRE(op != COBEL_OP_UPDATE_Q || (p->Q && p->lr && p->gamma), COBEL_EINVAL, "Q / lr / gamma missing");
  COBEL_REQUIRE(exp_ok(e, true), COBEL_EINVAL, "experience batch missing");
  COBEL_REQUIRE(!(p->mod_flags & COBEL_SFMA_MOD_REWARD) || p->D, COBEL_EINVAL, "reward_mod needs the similarity matrix");
  COBEL_DISPATCH_A(p->world.n_actions, (sfma_op_kernel<A><<<grid_for(p->n_agents), kT, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*p, op, *e)));
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}

extern "C" int cobel_pma_op(const CobelPMAParams* p, int op, const CobelExperiences* e, const int32_t* state, double* out, void* stream) {
  COBEL_REQUIRE(p && p->n_agents > 0 && p->world.n_states > 0, COBEL_EINVAL, "null / empty params");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (op == COBEL_OP_GAIN_BATCH) {
    COBEL_REQUIRE(out && p->Q && p->Mr && p->Ms && p->Mt && p->lr_q && p->gamma_q && p->mem_policy.param, COBEL_EINVAL, "cobel_pma_op(GAIN_BATCH): out[N, S*A] and the memory's parameters are needed");
    const int64_t total = p->n_agents * p->world.n_states * p->world.n_actions;
    COBEL_DISPATCH_A(p->world.n_actions, (pma_gain_batch_kernel<A><<<grid_for(total), kT, 0, st>>>(*p, out)));
  } else {
    COBEL_REQUIRE(op == COBEL_OP_STORE || op == COBEL_OP_UPDATE_Q || op == COBEL_OP_NEED, COBEL_EINVAL, "cobel_pma_op: unknown op %d", op);
    COBEL_REQUIRE(op == COBEL_OP_NEED ? (state && out && p->need_scratch && p->SR) : exp_ok(e, true), COBEL_EINVAL, "cobel_pma_op: arguments of the op missing");
    COBEL_REQUIRE(op != COBEL_OP_STORE || (p->Mr && p->Ms && p->Mt && p->T && p->mem_lr), COBEL_EINVAL, "memory tables / mem_lr missing");
    COBEL_REQUIRE(op != COBEL_OP_UPDATE_Q || (p->Q && p->lr && p->pow_gamma_q && e->batch <= COBEL_PMA_MAX_SEQ), COBEL_EINVAL,
                  "cobel_pma_op(UPDATE_Q): lr, pow_gamma_q (= agent.gamma ** k) and at most %d experiences", COBEL_PMA_MAX_SEQ);
    CobelExperiences none{};
    COBEL_DISPATCH_A(p->world.n_actions, (pma_op_kernel<A><<<grid_for(p->n_agents), kT, 0, st>>>(*p, op, e ? *e : none, state, out)));
  }
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}
