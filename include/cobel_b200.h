/*
 * cobel_b200.h -- C ABI of the B200-native batched tabular simulator.
 *
 * Drop-in boundary for CoBeL-RL's tabular closed loop (reference: sencheng/CoBeL-RL
 * v3.0.1, paths below are relative to src/cobel/).  The reference has no FFI: its
 * boundary is the Python class API.  Each entry point here replaces one
 * `Agent.train()/test()` loop of the reference for N independent agents and is
 * bound from Python with ctypes (cobel-rl_b200/_lib.py); INTEGRATION.md shows
 * the binding a maintainer of the reference would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless stated otherwise; the caller
 *    (PyTorch) owns all buffers, kernels never allocate or free;
 *  - all reals are IEEE fp64 and are combined in the reference's operation
 *    order without FMA contraction, so tables are bit-equal to NumPy's;
 *  - N = n_agents, S = n_states, A = n_actions; leading axis of every per-agent
 *    tensor is the agent; tensors are C-contiguous;
 *  - entry points return 0 on success or a negative COBEL_E* code;
 *    cobel_last_error() returns the message of the calling thread's last failure.
 *    Launches are asynchronous on `stream` (a cudaStream_t passed as void*).
 */
#ifndef COBEL_B200_H
#define COBEL_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COBEL_ABI_VERSION 6

enum {
  COBEL_OK = 0,
  COBEL_EINVAL = -1,      /* bad argument (the AssertionError / ValueError cases of the reference) */
  COBEL_EUNSUPPORTED = -2,/* shape outside what the kernels were built for */
  COBEL_ECUDA = -3        /* CUDA runtime error at launch */
};

/* Action-selection policies: policy/greedy.py:60-88 (EpsilonGreedy), 117-147
 * (ExclusiveEpsilonGreedy), policy/softmax.py:60-88 (Softmax). */
enum { COBEL_POLICY_EPS_GREEDY = 0, COBEL_POLICY_EXCL_EPS_GREEDY = 1, COBEL_POLICY_SOFTMAX = 2 };

/* Environment tables: interface/gridworld.py:92-145 (`sas` compiled to its arg-max
 * successor, rewards/terminals looked up at the arrival state) and
 * interface/topology.py:126-172 (`neighbors` lists). */
typedef struct CobelWorld {
  int32_t n_states;
  int32_t n_actions;
  int32_t n_starts;
  int32_t reserved;
  const int32_t* succ;      /* [S*A]  successor of (s,a) */
  const double*  reward;    /* [S]    reward on arrival */
  const uint8_t* terminal;  /* [S]    1 = trial ends on arrival */
  const int32_t* starts;    /* [K]    starting states, reset draws uniformly */
  /* Non-deterministic gridworlds (interface/gridworld.py:118-123): CSR of the non-zero entries of
   * sas[s,a,:] in ascending next-state order; the step then consumes one more uniform and draws
   * s' ~ categorical(sas[s,a,:]) exactly like Generator.choice(p=...).  NULL = deterministic (succ). */
  const int32_t* tp_off;    /* [S*A+1] */
  const int32_t* tp_next;   /* [nnz]   */
  const double*  tp_prob;   /* [nnz]   */
} CobelWorld;

/* Random-stream contract (one uniform stream per agent, consumed in program
 * order by environment, policies, memory and agent alike -- the reference run
 * with one shared numpy Generator).  Draw k of agent g is Philox4x32-10 with
 * key = seed, counter = (k>>1, g), 53-bit mantissa construction; see
 * oracle/philox.py.  If user_stream != NULL draws are read from it instead. */
typedef struct CobelStream {
  uint64_t seed;
  int64_t  agent_id_base;    /* global id of local agent 0 (multi-GPU shards) */
  int64_t* draw_count;       /* [N] in/out: number of draws consumed so far */
  const double* user_stream; /* optional [N, user_stream_len] uniforms in [0,1) */
  int64_t  user_stream_len;
} CobelStream;

typedef struct CobelPolicy {
  int32_t kind;              /* COBEL_POLICY_* */
  int32_t reserved;
  const double* param;       /* [N] epsilon or beta per agent */
} CobelPolicy;

/* Per-agent outputs that replace the reference's `logs` dict / callbacks
 * (agent/dyna_q.py:165-212).  Optional members may be NULL. */
typedef struct CobelTrace {
  int32_t* trial_steps;      /* [N, trials] logs['steps'] = index of the last step */
  double*  trial_reward;     /* [N, trials] logs['trial_reward'] */
  int64_t* n_steps;          /* [N] in/out: environment steps executed (accumulates) */
  int64_t* n_replay;         /* [N] in/out: replayed updates executed (accumulates) */
  int32_t* step_sa;          /* optional [N, step_cap]: s*A + a of every step */
  int64_t  step_cap;
  int32_t* replay_idx;       /* optional [N, replay_cap]: flat index of every replayed experience */
  int64_t  replay_cap;
  int32_t* replay_len;       /* optional [N, replay_calls_cap]: length of every replay call */
  int64_t  replay_calls_cap;
  int32_t* flags;            /* optional [N] in/out: COBEL_FLAG_* bits raised by the agent */
  int32_t* step_next;        /* optional [N, step_cap]: arrival state of every step (needed to reconstruct
                                trajectories in non-deterministic worlds) */
  double*  step_td;          /* optional [N, step_cap]: TD error of the online update of every step, the value
                                that feeds Q[s,a] += lr * td (Dyna-Q, QAgent, SFMA, PMA; ignored by the SR agents
                                and by runs that do not learn) */
  double*  replay_td;        /* optional [N, replay_cap], needs replay_idx: TD error of every replayed update, entry for
                                entry with replay_idx, the value that feeds Q[s,a] += lr * td (cobel_dynaq_run,
                                cobel_q_run, cobel_sfma_run, cobel_pma_run in a call that replays; PMA: the td of the
                                element that replay_idx names in its n-step update, NaN where that update aborted).
                                Entries of replays that update nothing (SFMA's trace-only replay at trial start) are
                                left untouched, as are all entries in the stand-alone entry points and the SR agents:
                                fill it with NaN to tell them apart.  NULL = not recorded.  It also pads the struct to
                                a multiple of 16 bytes: the members that follow an embedded CobelTrace keep their
                                16-byte alignment in the kernel parameter block */
} CobelTrace;

enum {
  COBEL_FLAG_TRACE_OVERFLOW = 1,  /* a step_sa / step_td / replay_idx / replay_td / replay_len buffer was too small */
  COBEL_FLAG_CDF_NEAR_TIE   = 2,  /* an inverse-CDF draw fell within rounding distance of a bin edge */
  COBEL_FLAG_LOG_OVERFLOW   = 4,  /* QAgent experience log full */
  COBEL_FLAG_SINGULAR       = 8,  /* PMA: (I - gamma T) pivot underflow */
  COBEL_FLAG_VISITED_OVERFLOW = 16,/* compact SR: an agent visited more than max_visited distinct states */
  COBEL_FLAG_BAND_VIOLATION = 32, /* PMA: T or a transition outside the band promised by sr_band */
  COBEL_FLAG_REPLAY_OVERFLOW = 64 /* SFMA: more experienced (s, a) than the replay kernel's on-chip list holds */
};

/* ---- Dyna-Q: agent/dyna_q.py:140-330 + memory/dyna_q.py:62-157 ------------- */
typedef struct CobelDynaQParams {
  int64_t n_agents;
  CobelWorld world;
  CobelStream stream;
  CobelPolicy policy;
  CobelTrace trace;
  double*  Q;                /* [N,S,A] agent.Q */
  double*  Mr;               /* [N,S,A] M.rewards */
  int32_t* Ms;               /* [N,S,A] M.states (init: self-loops) */
  int32_t* Mt;               /* [N,S,A] M.terminals (holds 1 - end_trial) */
  const uint8_t* action_mask;/* [S,A] or [N,S,A] (see mask_agent_stride); NULL = mask_actions False */
  int64_t  mask_agent_stride;/* 0 = one mask shared by all agents, S*A = per agent */
  const double* lr;          /* [N] agent.learning_rate */
  const double* gamma;       /* [N] agent.gamma */
  const double* mem_lr;      /* [N] M.learning_rate */
  int32_t trials, steps, batch;
  int32_t learn;             /* 1 = train(), 0 = test() (policy only; no store/update/replay) */
  int32_t no_replay;         /* train(..., no_replay=True) */
  int32_t episodic_replay;   /* agent.episodic_replay */
} CobelDynaQParams;

int cobel_dynaq_run(const CobelDynaQParams* p, void* stream);

/* ---- QAgent: agent/q.py:115-354 (tabular Q-learning, append-only experience log) -------- */
typedef struct CobelQParams {
  int64_t n_agents;
  CobelWorld world;          /* Gridworld tables or Topology graph (neighbors -> succ) */
  CobelStream stream;
  CobelPolicy policy;
  CobelTrace trace;          /* replay_idx holds log indices */
  double*  Q;                /* [N, n_keys, A] rows keyed by observation (agent.Q dict, q.py:142,197-204) */
  const int32_t* obs_key;    /* [S] node/state -> Q row; NULL = identity */
  int32_t  n_keys;
  int32_t  reserved;
  void*    log;              /* [N, log_cap] 16-byte records {f64 reward; u16 state, next_state; u8 action,
                                nonterminal; u16 pad} = agent.M (q.py:143,213) */
  int64_t  log_cap;
  int64_t* log_len;          /* [N] in/out: experiences stored so far */
  const double* lr;          /* [N] */
  const double* gamma;       /* [N] */
  int32_t trials, steps, batch;
  int32_t learn;             /* 1 = train(), 0 = test() */
} CobelQParams;

int cobel_q_run(const CobelQParams* p, void* stream);

/* ---- SR agent: agent/sr.py:109-324 (dense successor representation) ---------------------- */
typedef struct CobelSRParams {
  int64_t n_agents;
  CobelWorld world;
  CobelStream stream;
  CobelPolicy policy;
  CobelTrace trace;
  double*  SR;               /* [N,S,S] agent.SR (init: identity) */
  double*  rewards;          /* [N,S]   agent.rewards (learned reward per state) */
  int32_t* model;            /* [N,S,A] arg-max of agent.transitions[s,a,:] (init: s) */
  const uint8_t* action_mask;/* [S,A] or [N,S,A]; NULL = mask_actions False */
  int64_t  mask_agent_stride;
  const double* lr;          /* [N] */
  const double* gamma;       /* [N] */
  int32_t trials, steps;
  int32_t learn;             /* 1 = train(), 0 = test() */
  int32_t reserved;
} CobelSRParams;

int cobel_sr_run(const CobelSRParams* p, void* stream);

/* ---- SR agent with visited-set compaction (very large state spaces, config C5) --------------- */
typedef struct CobelSRCompactParams {
  int64_t n_agents;
  CobelWorld world;
  CobelStream stream;
  CobelPolicy policy;
  CobelTrace trace;
  double*  SRc;              /* [N,Vmax,Vmax] SRc[i,j] = agent.SR[visited[i], visited[j]]; rows/columns beyond
                                n_visited are undefined; every other entry of the dense SR is the identity */
  double*  rewards;          /* [N,Vmax] agent.rewards at the visited states (0 elsewhere) */
  int32_t* model;            /* [N,Vmax,A] LOCAL index of the modelled successor of (visited[i], a) (self elsewhere) */
  int32_t* visited;          /* [N,Vmax] global state of local index i, in order of first visit */
  int32_t* n_visited;        /* [N] in/out: V */
  const uint8_t* action_mask;/* [S,A] shared by all agents; NULL = mask_actions False */
  const double* lr;          /* [N] */
  const double* gamma;       /* [N] */
  int32_t max_visited;       /* Vmax, 2..65535.  Up to the on-chip limit (1309 / 1066 / 900 / 685 / 553 at 2 / 3 / 4 / 6 / 8
                                actions) visited / rewards / model are staged in shared memory; above it they stay in
                                HBM (one CTA per agent), limited only by the n_states slot map fitting in shared memory */
  int32_t trials, steps;
  int32_t learn;
} CobelSRCompactParams;

int cobel_sr_compact_run(const CobelSRCompactParams* p, void* stream);

/* ---- SFMA: agent/sfma.py:189-474 + memory/sfma.py:21-416 --------------------------------- */
enum { COBEL_SFMA_DEFAULT = 0, COBEL_SFMA_FORWARD = 1, COBEL_SFMA_REVERSE = 2, COBEL_SFMA_BLEND_FORWARD = 3,
       COBEL_SFMA_BLEND_REVERSE = 4, COBEL_SFMA_INTERPOLATE = 5, COBEL_SFMA_SWEEPING = 6 };

/* CobelSFMAParams.mod_flags (memory/sfma.py:216-236, 283-288, 319-320) */
#define COBEL_SFMA_MOD_REWARD_LOCAL 1   /* M.reward_mod_local: C[a,s] += r * reward_modulation on store */
#define COBEL_SFMA_MOD_REWARD       2   /* M.reward_mod: C += r * tile(D[s]) * reward_modulation on store */
#define COBEL_SFMA_MOD_STATE        4   /* M.state_mod: C[.,s] += 1 on store */
#define COBEL_SFMA_C_NORMALIZE      8   /* M.C_normalize */
#define COBEL_SFMA_D_NORMALIZE     16   /* M.D_normalize */
#define COBEL_SFMA_R_RAW           32   /* M.R_normalize == False */

typedef struct CobelSFMAParams {
  int64_t n_agents;
  CobelWorld world;
  CobelStream stream;
  CobelPolicy policy;
  CobelTrace trace;          /* replay_idx holds flat indices a*S + s; replay_len the length of each replay */
  double*  Q;                /* [N,S,A] */
  double*  Mr;               /* [N,S,A] M.rewards */
  int32_t* Ms;               /* [N,S,A] M.states (init: self-loops) */
  int32_t* Mt;               /* [N,S,A] M.terminals */
  double*  C;                /* [N,S*A] M.C experience strengths, index a*S + s */
  double*  T;                /* [N,S*A] M.T recency */
  double*  I;                /* [N,S]   M.I inhibition */
  const double* D;           /* [S,S]   metric.D similarity matrix, shared by all agents */
  const uint8_t* action_mask;/* [S,A] or [N,S,A]; NULL = mask_actions False */
  int64_t  mask_agent_stride;
  const double* lr;          /* [N] agent.learning_rate */
  const double* gamma;       /* [N] agent.gamma */
  const double* mem_lr;      /* [N] M.learning_rate */
  double beta;               /* M.beta (20) */
  double threshold;          /* M.R_threshold (1e-6) */
  double decay_inhibition;   /* M.decay_inhibition (0.9) */
  double decay_strength;     /* M.decay_strength (1.0) */
  double decay_recency;      /* M.decay_recency (0.9) */
  double c_step, i_step;     /* M.C_step, M.I_step (1.0) */
  double blend, interp_fwd, interp_rev;   /* M.blend, M.interpolation_fwd / _rev */
  int32_t mode;              /* COBEL_SFMA_* (M.mode) */
  int32_t recency;           /* M.recency */
  int32_t deterministic;     /* M.deterministic */
  int32_t trials, steps, batch;
  int32_t nb_replays;        /* agent.nb_replays */
  int32_t start_replay;      /* agent.start_replay */
  int32_t random_replay;     /* agent.random: uniform batches over the unmasked experiences (memory/sfma.py:375-416) */
  int32_t dynamic;           /* agent.dynamic: 'reverse' / 'default' chosen per trial from td_acc (agent/sfma.py:311-318) */
  int32_t no_replay;
  int32_t learn;             /* 1 = train(), 0 = test() */
  double*  td_acc;           /* optional [N] in/out: agent.td, the |TD error| accumulated by update_q (agent/sfma.py:456) */
  int32_t* trial_mode;       /* optional [N,trials] out: replay mode chosen at the end of each trial (dynamic) */
  double   reward_modulation;/* M.reward_modulation (1.0) */
  int32_t  mod_flags;        /* COBEL_SFMA_MOD_* bits: strength modulation and normalisation switches */
  int32_t  exp_bound;        /* 1 + an upper bound on the number of (s, a) with C > 0 that any agent holds when the call starts; 0 =
                                unknown.  The split path sizes the replay kernel's on-chip list by exp_bound - 1 + the steps taken
                                so far instead of S*A: less shared memory per agent, more agents per SM */
  int64_t* carry;            /* scratch [N,4], required: per-agent state between the launches of the split path (one
                                thread per agent for the online steps, one CTA per agent for the replays) */
  uint8_t* workspace;        /* scratch [N, cobel_sfma_workspace_bytes(p)]: the fused kernel's per-agent tables when they
                                exceed shared memory; may be NULL when the query returns 0 */
} CobelSFMAParams;

int cobel_sfma_run(const CobelSFMAParams* p, void* stream);
/* Bytes of CobelSFMAParams.workspace per agent that cobel_sfma_run needs for this configuration: 0 when it takes the
 * split path (decay_strength == 1, M.T neither read (recency) nor kept (train(no_replay=True)), no reward_mod) or when
 * the fused kernel's per-agent tables fit in shared memory; else the size of those tables, which then live in the
 * workspace.  Reads n_states, n_actions, batch, recency, no_replay, learn, decay_strength, mod_flags, random_replay.
 * Negative COBEL_E* code on bad arguments (more than 32767 states: COBEL_EUNSUPPORTED). */
int64_t cobel_sfma_workspace_bytes(const CobelSFMAParams* p);

/* ---- PMA: agent/pma.py:137-369 + memory/pma.py:20-496 (Mattar & Daw gain x need replay) ---- */
#define COBEL_PMA_MAX_SEQ 64      /* longest n-step sequence = largest replay batch */
/* CobelPMAParams.options (memory/pma.py:238-249) */
#define COBEL_PMA_OPT_EQUAL_NEED    1   /* M.equal_need: need.fill(1) */
#define COBEL_PMA_OPT_EQUAL_GAIN    2   /* M.equal_gain: gain.fill(1) */
#define COBEL_PMA_OPT_KEEP_BARRIERS 4   /* M.ignore_barriers == False: utility is not multiplied by update_mask */
#define COBEL_PMA_OPT_ALLOW_LOOPS   8   /* M.allow_loops: a sequence is extended even if it revisits a state */

typedef struct CobelPMAParams {
  int64_t n_agents;
  CobelWorld world;
  CobelStream stream;
  CobelPolicy policy;        /* agent.policy (online action selection) */
  CobelPolicy mem_policy;    /* M.policy (gain evaluation and sequence extension) */
  CobelTrace trace;          /* replay_idx holds flat indices a*S + s of the performed updates */
  double*  Q;                /* [N,S,A] */
  double*  Mr;               /* [N,S,A] M.rewards */
  int32_t* Ms;               /* [N,S,A] M.states (init: 0, memory/pma.py:136) */
  int32_t* Mt;               /* [N,S,A] M.terminals */
  double*  T;                /* [N,S,S] M.T learned state-state transition matrix */
  double*  SR;               /* [N,S,S] M.SR = inv(I - gamma T), refreshed every trial */
  const uint8_t* update_mask;/* [N,S*A] M.update_mask, index a*S + s */
  const uint8_t* action_mask;/* [S,A] or [N,S,A]; NULL = mask_actions False */
  int64_t  mask_agent_stride;
  const double* lr;          /* [N] agent.learning_rate */
  const double* gamma;       /* [N] agent.gamma */
  const double* mem_lr;      /* [N] M.learning_rate */
  const double* lr_q;        /* [N] M.learning_rate_q */
  const double* gamma_q;     /* [N] M.gamma_q */
  const double* gamma_sr;    /* [N] M.gamma */
  const double* pow_gamma_sr;/* [COBEL_PMA_MAX_SEQ+2] (or per agent, see pow_stride): float(M.gamma) ** k */
  const double* pow_gamma_q; /* same for M.gamma_q (the reference uses Python's float pow) */
  int64_t  pow_stride;       /* 0 = one table for all agents, COBEL_PMA_MAX_SEQ+2 = one per agent */
  double*  min_gap;          /* optional [N] in/out: smallest relative gap between the two largest distinct utilities */
  int64_t* carry;            /* scratch [N,8]: per-agent state carried between the launches of one call */
  double*  need_scratch;     /* scratch [2,N,S]: the `need` vector of the next replay call (an SR row from the banded solve or the
                                stationary distribution of a timed-out trial); second plane: SR[start] of the next trial */
  double   lr_T;             /* M.learning_rate_T (0.9) */
  double   min_gain;         /* M.min_gain (1e-6) */
  int32_t  min_gain_original;/* M.min_gain_mode == 'original' */
  int32_t trials, steps, batch;
  int32_t no_replay;
  int32_t learn;             /* 1 = train(), 0 = test() */
  /* Banded update_sr (memory/pma.py:413-415 needs only the SR rows that replay reads, :401-411).  sr_band in 0..31 is
   * the caller's guarantee that T[i][j] == 0 for |i - j| > sr_band and that every world transition satisfies
   * |s' - s| <= sr_band (a W-wide gridworld: sr_band = W): each agent then factorises its banded I - gamma T after
   * every trial (its own kernels between the phases of the main kernel) and solves for the one SR row a replay call needs, and SR is refreshed
   * once, densely, at the end of the call.  A violated guarantee raises COBEL_FLAG_BAND_VIOLATION.
   * sr_band < 0: dense update_sr after every trial (any T). */
  int32_t sr_band;
  int32_t options;           /* COBEL_PMA_OPT_* bits */
  double*  band_scratch;     /* scratch [N, S*(2*sr_band+1)] when sr_band >= 0 (the band factors of I - gamma T) */
  /* Tie-pattern policy tables (optional, A <= 4, the two epsilon-greedy kinds).  get_action_probs of those
   * policies (policy/greedy.py:60-88,117-147) depends only on which actions are valid and which of them tie for
   * the row maximum, so raw probabilities, action_probs_batch's p / sum(p) (memory/pma.py:423-450) and
   * select_action's cumsum(p) / cumsum(p)[-1] (policy/greedy.py:58) are tabulated once per distinct
   * (kind, parameter) -- with exactly the per-row operations -- and a gain evaluation becomes a row maximum,
   * A compares and one table row.  n_tab = 0: probabilities are evaluated per row (any policy, any A). */
  int32_t  n_tab;            /* number of tables */
  int32_t  band_trusted;     /* 1: the caller vouches that the initial T lies inside sr_band (e.g. it was left by a previous call of this
                                library, which enforces the band on every transition) -- the streaming check of T is skipped */
  const int32_t* tab_kind;   /* [n_tab] COBEL_POLICY_* of table t (a Softmax entry leaves its table unused) */
  const double*  tab_param;  /* [n_tab] its epsilon */
  const int32_t* tab_of_agent;/* optional [N,2]: tables of (agent.policy, M.policy) of agent n; NULL = (0, n_tab-1) */
  double*  tab_scratch;      /* scratch [n_tab * COBEL_PMA_TAB_DOUBLES(A) + COBEL_PMA_TIE_DOUBLES], filled by the call (the
                                tail holds the bin edges of Generator.choice over k <= 32 tied utilities) */
} CobelPMAParams;
#define COBEL_PMA_TAB_DOUBLES(A) (3 * (1 << (2 * (A))) * (A))
#define COBEL_PMA_TIE_DOUBLES 1024

int cobel_pma_run(const CobelPMAParams* p, void* stream);

/* ---- stand-alone methods ------------------------------------------------------------------------------------
 * One call = one method of the reference's classes for all N agents, for callers that drive the loop themselves
 * (env.step -> policy.select_action -> M.store -> agent.update_q -> agent.replay, agent/dyna_q.py:176-203) instead
 * of the fused train().  Same arithmetic, same stream contract; one thread per agent (csrc/ops.cu), the two
 * replay generators are phases of the fused kernels. */

/* B experiences per agent, [N,B] each: the Experience dicts of memory/dyna_q.py:8-14, agent/q.py:17-23,
 * agent/sr.py:16-22, memory/pma.py:11-17, memory/sfma.py:12-18 as a structure of arrays. */
typedef struct CobelExperiences {
  int32_t  batch;            /* B */
  int32_t  reserved;
  int32_t* state;            /* [N,B] */
  int32_t* action;           /* [N,B] */
  double*  reward;           /* [N,B] */
  int32_t* next_state;       /* [N,B] */
  int32_t* terminal;         /* [N,B] holds 1 - end_trial, like the reference's field of that name */
  double*  td;               /* optional [N,B]: out, the TD error update_q adds to the dict */
} CobelExperiences;

enum {
  COBEL_OP_STORE = 1,          /* Memory.store(e[.,0]) / QAgent: M.append / SR: SR.update(e[.,0]) */
  COBEL_OP_UPDATE_Q = 2,       /* Agent.update_q for the B experiences in order (PMA: the batch is ONE n-step update) */
  COBEL_OP_RETRIEVE_BATCH = 3, /* DynaQMemory.retrieve_batch(B) -> e */
  COBEL_OP_REPLAY = 4,         /* Agent.replay(B): draw, then update_q in order; e receives the batch */
  COBEL_OP_RETRIEVE_Q = 5,     /* SR.retrieve_q(state) -> q_out[N,A] */
  COBEL_OP_GATHER = 6,         /* SFMA: e.state holds flat indices a*S+s (-1 = none); fills e with the stored experiences */
  COBEL_OP_GAIN_BATCH = 7,     /* PMAMemory.compute_gain_batch -> out[N,S*A] */
  COBEL_OP_NEED = 8            /* PMAMemory.compute_need(state) -> out[N,S*A]; state < 0: need_scratch (stationary) tiled */
};

/* Interface.reset() / Interface.step(action): interface/gridworld.py:92-145, interface/topology.py:126-172.
 * state[N] in/out (reset: out), reward[N], end_trial[N] out. */
int cobel_env_reset(const CobelWorld* w, const CobelStream* s, int64_t n_agents, int32_t* state, void* stream);
int cobel_env_step(const CobelWorld* w, const CobelStream* s, int64_t n_agents, int32_t* state, const int32_t* action,
                   double* reward, uint8_t* end_trial, void* stream);
/* Policy.get_action_probs(values[., A], mask) for rows_per_agent rows per agent, and Policy.select_action (one row and one
 * draw per agent): policy/greedy.py:40-147, policy/softmax.py:40-88.  mask: [rows, A] bytes or NULL. */
int cobel_policy_probs(const CobelPolicy* pol, int64_t n_agents, int64_t rows_per_agent, int32_t n_actions,
                       const double* values, const uint8_t* mask, double* probs, void* stream);
int cobel_policy_select(const CobelPolicy* pol, const CobelStream* s, int64_t n_agents, int32_t n_actions,
                        const double* values, const uint8_t* mask, int32_t* action, void* stream);
/* DynaQMemory.store / retrieve_batch, DynaQ.update_q / replay: memory/dyna_q.py:77-157, agent/dyna_q.py:275-330 */
int cobel_dynaq_op(const CobelDynaQParams* p, int op, const CobelExperiences* e, void* stream);
/* QAgent: M.append (STORE), update_q, replay (e.state receives the replayed log indices): agent/q.py:205-215, 297-354 */
int cobel_q_op(const CobelQParams* p, int op, const CobelExperiences* e, void* stream);
/* SR.update (STORE) / SR.retrieve_q: agent/sr.py:255-308 */
int cobel_sr_op(const CobelSRParams* p, int op, const CobelExperiences* e, const int32_t* state, double* q_out, void* stream);
/* SR.update (STORE: e[.,0] per agent) / SR.retrieve_q for B states per agent (RETRIEVE_Q: states[N,B] -> q_out[N,B,A])
 * on the compact tables of cobel_sr_compact_run.  Consumes no draws.  One launch per call, one CTA per agent
 * (csrc/sr_compact.cu); reads SRc / rewards / model / visited / n_visited / lr / gamma / max_visited /
 * world.n_states / world.n_actions / n_agents and, of the trace, only flags.  STORE locates or inserts s, then s',
 * exactly like a learning step of train() (an insertion beyond max_visited raises COBEL_FLAG_VISITED_OVERFLOW in
 * trace.flags); RETRIEVE_Q inserts nothing and is bit-identical to cobel_sr_op on the dense tables.  Every state
 * must lie in 0..S-1.  COBEL_EUNSUPPORTED when the slot map of S states (and, for RETRIEVE_Q, a list of up to
 * min(max_visited, S) columns) does not fit in shared memory. */
int cobel_sr_compact_op(const CobelSRCompactParams* p, int op, const CobelExperiences* e, const int32_t* states,
                        int32_t n_query, double* q_out, void* stream);
/* SFMAMemory.store, SFMA.update_q (learn = 0: no_update), GATHER: memory/sfma.py:195-236, agent/sfma.py:423-458 */
int cobel_sfma_op(const CobelSFMAParams* p, int op, const CobelExperiences* e, void* stream);
/* SFMAMemory.replay(batch, state) [apply_updates = 0] / SFMA.replay(batch, state) [apply_updates = 1] /
 * SFMAMemory.retrieve_random_batch(batch, mask) [apply_updates = 2, random_replay = 1]
 * (memory/sfma.py:238-347, 375-416, agent/sfma.py:392-421): state[N] = current state, -1 = None.  The reactivated
 * flat indices go to trace.replay_idx / replay_len (mandatory here); needs p.carry.  recency = 1 weights the priority by
 * M.T (p.T), as train() does. */
int cobel_sfma_replay(const CobelSFMAParams* p, const int32_t* state, int apply_updates, void* stream);
/* PMAMemory.store, PMA.update_q (pow_gamma_q must hold agent.gamma ** k), compute_gain_batch, compute_need:
 * memory/pma.py:148-166, 333-411, agent/pma.py:319-353 */
int cobel_pma_op(const CobelPMAParams* p, int op, const CobelExperiences* e, const int32_t* state, double* out, void* stream);
/* PMAMemory.replay(Q, action_mask, batch, state) (memory/pma.py:168-267): state[N] = current state, -1 = None (the
 * need is then the stationary distribution of T).  Q is updated in place, the performed updates go to
 * trace.replay_idx / replay_len.  update_sr != 0: M.update_sr() first (memory/pma.py:413-415), then the need from the
 * refreshed SR.  At most 512 states and 2048 one-step backups.  Up to 160 states and 1024 backups SR and the
 * stationary need come from the dense eliminations (sr_band is ignored).  Beyond either bound the banded ones are
 * used, so sr_band must be 0..31 with band_scratch (else COBEL_EUNSUPPORTED): the band LU of I - gamma T and the full
 * SR refresh for update_sr, the banded GTH for the agents whose state is -1.  band_trusted = 0 checks T against the
 * band first (COBEL_FLAG_BAND_VIOLATION).  Every size is checked before the first launch. */
int cobel_pma_replay(const CobelPMAParams* p, const int32_t* state, int update_sr, void* stream);

/* ---- utilities -------------------------------------------------------------- */
int  cobel_abi_version(void);
/* Copy the last error message of this thread into buf (NUL-terminated). */
void cobel_last_error(char* buf, size_t len);
/* Fill out[N, n_draws] with draws first..first+n_draws-1 of agents
 * agent_id_base..+N-1 (device buffer).  Used to check the stream contract. */
int  cobel_draw_uniforms(uint64_t seed, int64_t agent_id_base, int64_t n_agents,
                         int64_t first, int64_t n_draws, double* out, void* stream);
/* Draw the next n_draws uniforms of every agent at its own draw_count (out[N, n_draws], device)
 * and advance draw_count -- serves Interface.reset()/Policy.select_action() outside train(). */
int  cobel_stream_next(const CobelStream* s, int64_t n_agents, int64_t n_draws, double* out, void* stream);
/* sizeof() of an ABI struct by name ("CobelDynaQParams", ...), 0 if unknown: lets a binding
 * verify its mirror of the layout. */
size_t cobel_sizeof(const char* struct_name);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t cobel_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* COBEL_B200_H */
