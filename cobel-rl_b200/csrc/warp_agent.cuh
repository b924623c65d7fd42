// warp_agent.cuh -- building blocks shared by the warp-per-agent kernels (Dyna-Q, QAgent, SFMA...):
// a 64-draw window of the agent's Philox stream generated lane-parallel, warp-uniform action
// selection with the (few) fp64 divisions spread over lanes, and the conflict-free
// level-parallel execution of a batch of sequential one-step TD updates.
#pragma once
#include "common.cuh"

constexpr unsigned kFull = 0xffffffffu;

COBEL_DEV double shfl_f64(double v, int src) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_sync(kFull, lo, src);
  hi = __shfl_sync(kFull, hi, src);
  return __hiloint2double(hi, lo);
}

COBEL_DEV double shfl_f64_up(double v, int delta) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_up_sync(kFull, lo, delta);
  hi = __shfl_up_sync(kFull, hi, delta);
  return __hiloint2double(hi, lo);
}

COBEL_DEV double shfl_f64_xor(double v, int m) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_xor_sync(kFull, lo, m);
  hi = __shfl_xor_sync(kFull, hi, m);
  return __hiloint2double(hi, lo);
}

// Row of A doubles from a 16-byte aligned table (A even -> LDS.128 / LDG.128).
template <int A>
COBEL_DEV void load_row(const double* r, double (&v)[A]) {
  if constexpr (A % 2 == 0) {
#pragma unroll
    for (int x = 0; x < A; x += 2) {
      const double2 t = *reinterpret_cast<const double2*>(r + x);
      v[x] = t.x; v[x + 1] = t.y;
    }
  } else {
#pragma unroll
    for (int x = 0; x < A; ++x) v[x] = r[x];
  }
}

// Next state of a non-deterministic gridworld: Generator.choice(arange(S), p=sas[s,a,:])
// (interface/gridworld.py:118-123) = first index whose sequential cumsum / total exceeds u; the
// zero entries of the row add exact zeros, so the cumsum runs over the non-zeros only.
COBEL_DEV int stochastic_successor(const CobelWorld& w, int sa, double u) {
  const int lo = __ldg(w.tp_off + sa), hi = __ldg(w.tp_off + sa + 1);
  double tot = 0.0;
  for (int j = lo; j < hi; ++j) tot = xadd(tot, __ldg(w.tp_prob + j));
  double c = 0.0;
  for (int j = lo; j < hi; ++j) {
    c = xadd(c, __ldg(w.tp_prob + j));
    if (xdiv(c, tot) > u) return __ldg(w.tp_next + j);
  }
  return __ldg(w.tp_next + hi - 1);
}

// ---------------------------------------------------------------------------
// DrawWindow: lane l holds draws 2*(b0+l) and 2*(b0+l)+1 of the agent's stream, i.e. the warp
// holds the 64 consecutive draws starting at 2*b0.  One Philox block per lane per refill
// instead of one per draw per agent.
// ---------------------------------------------------------------------------
// One Philox block -> two uniforms, as ONE shared copy of the ~110-instruction sequence: for kernels that are
// instruction-fetch bound (PMA) and refill from several sites.
static __device__ __noinline__ double2 philox_pair_shared(uint64_t b, uint64_t agent, uint32_t key0, uint32_t key1) {
  uint32_t o[4];
  philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), (uint32_t)agent, (uint32_t)(agent >> 32), key0, key1, o);
  return make_double2(u53(o[0], o[1]), u53(o[2], o[3]));
}

// MAYBE_USER = false compiles the user-stream ("stream from HBM") branches out; SMALL_CODE = true refills
// through the shared (not inlined) Philox routine.
template <bool MAYBE_USER, bool SMALL_CODE = false>
struct DrawWindowT {
  uint64_t agent;
  uint32_t key0, key1;
  uint64_t base;          // stream index of window slot 0 (even)
  int off;                // window slot of the next draw: k = base + off
  int cap;                // slots filled (0 = empty, 64 after a refill)
  double ua, ub;          // this lane's two draws: slots 2*lane and 2*lane+1
  const double* user;     // optional pre-drawn stream of this agent
  int64_t user_len;

  COBEL_DEV void init(const CobelStream& s, int64_t local_agent, uint64_t k) {
    agent = (uint64_t)(s.agent_id_base + local_agent);
    key0 = (uint32_t)s.seed; key1 = (uint32_t)(s.seed >> 32);
    user = (MAYBE_USER && s.user_stream) ? s.user_stream + local_agent * s.user_stream_len : nullptr;
    user_len = s.user_stream_len;
    base = k; off = 0; cap = 0;     // empty: the first ensure() refills
    ua = ub = 0.0;
  }
  COBEL_DEV uint64_t position() const { return base + (uint64_t)off; }
  // make the next `need` draws available (need <= 63); warp-uniform
  COBEL_DEV void ensure(int need, int lane) {
    if ((MAYBE_USER && user) || off + need <= cap) return;
    const uint64_t k = base + (uint64_t)off;
    base = k & ~1ull; off = (int)(k & 1ull); cap = 64;
    const uint64_t b = (base >> 1) + lane;
    if constexpr (SMALL_CODE) {
      const double2 d = philox_pair_shared(b, agent, key0, key1);
      ua = d.x; ub = d.y;
    } else {
      uint32_t o[4];
      philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), (uint32_t)agent, (uint32_t)(agent >> 32), key0, key1, o);
      ua = u53(o[0], o[1]); ub = u53(o[2], o[3]);
    }
  }
  // draw number (next + ahead), `ahead` may differ per lane; all 32 lanes must call
  COBEL_DEV double peek(int ahead) const {
    if (MAYBE_USER && user) {
      const uint64_t kk = base + (uint64_t)(off + ahead);
      return kk < (uint64_t)user_len ? user[kk] : 0.0;
    }
    const int slot = off + ahead;
    const double a = shfl_f64(ua, slot >> 1), b = shfl_f64(ub, slot >> 1);
    return (slot & 1) ? b : a;
  }
  COBEL_DEV void advance(int n) { off += n; }
  COBEL_DEV double next() { const double u = peek(0); ++off; return u; }
  COBEL_DEV void attach(double*) {}
};
using DrawWindow = DrawWindowT<true>;

// ---------------------------------------------------------------------------
// SmemDrawWindow: the same interface over a window of kSmemDraws draws in shared memory (the PLAIN
// kernels).  A refill costs one Philox block per lane per 64 draws whatever is consumed, and a Dyna-Q
// step consumes 34: a 64-draw window serves one step per refill (53 % of the generated draws used), a
// 256-draw window seven (93 %); reading a draw is one LDS.64 instead of four shuffles.
// ---------------------------------------------------------------------------
constexpr int kSmemDraws = 256;
template <int NDRAWS>
struct SmemDrawWindowT {
  uint64_t agent;
  uint32_t key0, key1;
  uint64_t base;          // stream index of buf[0] (even)
  int off;                // buf slot of the next draw: k = base + off
  int cap;                // slots filled (0 = empty)
  double* buf;            // [NDRAWS], 16-byte aligned, this agent's

  COBEL_DEV void attach(double* b) { buf = b; }
  COBEL_DEV void init(const CobelStream& s, int64_t local_agent, uint64_t k) {
    agent = (uint64_t)(s.agent_id_base + local_agent);
    key0 = (uint32_t)s.seed; key1 = (uint32_t)(s.seed >> 32);
    base = k; off = 0; cap = 0;
  }
  COBEL_DEV uint64_t position() const { return base + (uint64_t)off; }
  COBEL_DEV void ensure(int need, int lane) {
    if (off + need <= cap) return;
    const uint64_t k = base + (uint64_t)off;
    base = k & ~1ull; off = (int)(k & 1ull); cap = NDRAWS;
    __syncwarp();                                   // every lane has read what it needed of the old window
#pragma unroll
    for (int j = 0; j < NDRAWS / 64; ++j) {
      const uint64_t b = (base >> 1) + (uint64_t)(j * 32 + lane);
      uint32_t o[4];
      philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), (uint32_t)agent, (uint32_t)(agent >> 32), key0, key1, o);
      reinterpret_cast<double2*>(buf)[j * 32 + lane] = make_double2(u53(o[0], o[1]), u53(o[2], o[3]));
    }
    __syncwarp();
  }
  COBEL_DEV double peek(int ahead) const { return buf[off + ahead]; }
  COBEL_DEV void advance(int n) { off += n; }
  COBEL_DEV double next() { return buf[off++]; }
};
using SmemDrawWindow = SmemDrawWindowT<kSmemDraws>;
template <bool PLAIN, int NDRAWS = kSmemDraws> struct WindowFor { using type = DrawWindowT<true>; };
template <int NDRAWS> struct WindowFor<true, NDRAWS> { using type = SmemDrawWindowT<NDRAWS>; };

// ---------------------------------------------------------------------------
// Warp-uniform action selection (all lanes hold the same v[], mask, u and get the same action).
//   probabilities: policy/greedy.py:60-88, 117-147; policy/softmax.py:60-88
//   draw: searchsorted(cumsum(p)/cumsum(p)[-1], u, 'right')   (policy/greedy.py:58)
// PolicyTab caches, per agent, the quotients eps/n and (1-eps)/n for n = 1..A in lane n-1.
// ---------------------------------------------------------------------------
struct PolicyTab {
  int kind;
  double par;
  double q_par;   // lane l: par / (l+1)
  double q_om;    // lane l: (1 - par) / (l+1)
  COBEL_DEV void init(int kind_, double par_, int lane) {
    kind = kind_; par = par_;
    q_par = xdiv(par_, (double)(lane + 1));
    q_om = xdiv(xsub(1.0, par_), (double)(lane + 1));
  }
};

// KIND >= 0 fixes the policy kind at compile time (drops the other kinds' code from the kernel)
template <int A, int KIND = -1>
COBEL_DEV int select_action_warp(const double (&v)[A], uint32_t mask, const PolicyTab& pt, double u, int lane) {
  const int kind = KIND >= 0 ? KIND : pt.kind;
  constexpr uint32_t kAll = (1u << A) - 1u;
  double m;
  int nv = A;
  if (mask == kAll) {
    m = row_max<A>(v);
  } else {
    nv = __popc(mask);
    m = -__longlong_as_double(0x7FF0000000000000ll);
#pragma unroll
    for (int a = 0; a < A; ++a) m = (mask >> a & 1u) ? xmax(m, v[a]) : m;
  }
  double p[A];
  if (kind == COBEL_POLICY_SOFTMAX) {
    double sum = 0.0;
#pragma unroll
    for (int a = 0; a < A; ++a) {
      p[a] = 0.0;
      if (mask >> a & 1u) { p[a] = exp(xmul(xsub(v[a], m), pt.par)); sum = xadd(sum, p[a]); }
    }
    if (A == 8 && mask == kAll) sum = np_sum<A>(p);        // np.sum over exactly 8 values is a tree, not a loop
#pragma unroll
    for (int a = 0; a < A; ++a)
      if (mask >> a & 1u) p[a] = xdiv(p[a], sum);
  } else {
    uint32_t ties = 0;
#pragma unroll
    for (int a = 0; a < A; ++a) ties |= (v[a] == m ? 1u : 0u) << a;
    ties &= mask;
    const int k = __popc(ties);
    const double tie = shfl_f64(pt.q_om, k - 1);                      // (1-eps)/k
    if (kind == COBEL_POLICY_EPS_GREEDY) {
      const double base = shfl_f64(pt.q_par, nv - 1);                 // eps/n_valid
      const double top = xadd(base, tie), low = xadd(base, 0.0);
#pragma unroll
      for (int a = 0; a < A; ++a)
        p[a] = (mask >> a & 1u) ? ((ties >> a & 1u) ? top : low) : 0.0;
    } else {
      const int d = nv - k > 1 ? nv - k : 1;
      const double expl = shfl_f64(pt.q_par, d - 1);                  // eps/max(n_valid-k,1)
      const double top = xadd(tie, 0.0), low = xadd(0.0, expl);
#pragma unroll
      for (int a = 0; a < A; ++a)
        p[a] = (mask >> a & 1u) ? ((ties >> a & 1u) ? top : low) : 0.0;
    }
  }
  // inverse CDF: lane a tests cdf[a]/cdf[A-1] <= u -- one division per lane instead of A-1 in
  // series, and none when the total is exactly 1.0 (x/1.0 == x)
  double c = p[0], mine = p[0];
#pragma unroll
  for (int a = 1; a < A; ++a) { c = xadd(c, p[a]); if (lane == a) mine = c; }
  if (c != 1.0) mine = xdiv(mine, c);
  const bool le = (lane < A - 1) && (mine <= u);
  return __popc(__ballot_sync(kFull, le));
}

// ---------------------------------------------------------------------------
// Epsilon-greedy over an unmasked row of A <= 4 actions: p[] (policy/greedy.py:60-88) depends only on
// the tie pattern (which entries equal the row maximum), so the 2^A - 1 possible normalised CDFs
// (policy/greedy.py:58) are tabulated once per agent -- with exactly the operations
// select_action_warp performs per step -- and a step is a row max, A compares and one lookup.
// `tab` is kEpsTabDoubles doubles of shared memory per agent: entry [pattern * 4 + a].
// ---------------------------------------------------------------------------
constexpr int kEpsTabDoubles = 64;
template <int A>
COBEL_DEV void eps_cdf_table_init(double* tab, const PolicyTab& pt, int lane) {
  static_assert(A <= 4, "tie-pattern table is built for at most 4 actions");
  const int pat = lane & ((1 << A) - 1);
  const int k = __popc(pat);
  const double base = shfl_f64(pt.q_par, A - 1);                    // eps/A
  const double tie = shfl_f64(pt.q_om, k > 0 ? k - 1 : 0);          // (1-eps)/k
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
  if (lane > 0 && lane < (1 << A)) {
#pragma unroll
    for (int a = 0; a < 4; ++a) tab[pat * 4 + a] = a < A ? cdf[a] : 2.0;
  }
  __syncwarp();
}
// bit a set = v[a] equals the row maximum m
template <int A>
COBEL_DEV uint32_t tie_pattern(const double (&v)[A], double m) {
  uint32_t ties = 0;
#pragma unroll
  for (int a = 0; a < A; ++a) ties |= (v[a] == m ? 1u : 0u) << a;
  return ties;
}
template <int A>
COBEL_DEV int select_action_eps_pattern(uint32_t ties, const double* tab, double u, int lane) {
  const double mine = tab[ties * 4 + (lane & 3)];
  return __popc(__ballot_sync(kFull, lane < A - 1 && mine <= u));
}
template <int A>
COBEL_DEV int select_action_eps_tab(const double (&v)[A], const double* tab, double u, int lane) {
  return select_action_eps_pattern<A>(tie_pattern<A>(v, row_max<A>(v)), tab, u, lane);
}

// ---------------------------------------------------------------------------
// Row summaries of an on-chip Q table (the PLAIN Dyna-Q kernel, A <= 4): V[s] = row_max(Q[s,:]) and
// P[s] = tie_pattern(Q[s,:]), computed with exactly the per-step operations, so reading them is bit-identical to
// recomputing them from the row.  Whoever writes Q[s,:] refreshes them before the next warp barrier.
// ---------------------------------------------------------------------------
template <int A>
COBEL_DEV void refresh_row_summary(const double* Q, double* V, uint8_t* P, int s) {
  double row[A];
  load_row<A>(Q + s * A, row);
  const double m = row_max<A>(row);
  V[s] = m;
  P[s] = (uint8_t)tie_pattern<A>(row, m);
}

// ---------------------------------------------------------------------------
// Level-parallel execution of a batch of one-step TD updates that the reference applies
// strictly in order (agent/dyna_q.py:329-330, agent/q.py:353-354).
//
// Lane j holds update j: it reads row Q[s2_j,:] and entry Q[s_j,a_j] and writes Q[s_j,a_j].
// For i < j:   i writes what j reads or writes  -> j must run in a LATER round
//              j writes what i reads            -> j must not run in an EARLIER round; the same round would do
//              (every round reads, syncs, then writes), but finding the largest such set needs a fixpoint loop
//              of ballots per round -- treating it like the first kind costs a few more rounds and measured 7 %
//              faster (one ballot per round).
// Rounds execute all currently ready lanes at once; each update sees exactly the values it
// would see in sequential order, so the result is bit-identical to the sequential loop.
//
// Most replayed updates leave Q bit-identical (early on most of the table is still 0; with a large
// learning rate in a deterministic world the entries soon reach exact fixed points), so every lane
// first evaluates its update against the pre-batch table without writing ("speculative pass"), and
// the updates that provably change nothing are dropped before the rounds:
//   null j  = the speculative Q[s_j,a_j] + lr*td has the same bits as Q[s_j,a_j];
//   valid j = every earlier update that writes what j reads (row s2_j, entry (s_j,a_j)) is valid and null.
// A valid j reads the pre-batch values in sequential order too, so its speculative value is its true
// value; if it is also null it writes what is already there, and removing it from the sequence changes
// no read or write before or after it.  If every lane is null, every lane is valid (induction from
// lane 0) and the batch is a no-op: no dependency analysis at all.  Otherwise the rounds run on the
// kept updates only, and the first round -- kept lanes whose dependences were all dropped, so their
// inputs are pre-batch values -- commits the speculative values without reloading.
// `wm`/`rm` are per-agent scratch arrays of S words in shared memory, zero between calls.
// ---------------------------------------------------------------------------
// `mbits` (optional) holds one byte per state with bit a set = action a may enter the max over
// Q[s2,:] (SFMA.update_q honours the action mask, agent/sfma.py:440-449; DynaQ / QAgent do not).
// `td_out` (optional): receives this lane's TD error (SFMA accumulates |td|, agent/sfma.py:456).
// SUM: the table keeps row summaries `V`/`P` (refresh_row_summary).  The speculative pass reads V[s2] (one LDS.64)
// instead of the row; the rounds keep reading rows, because V is stale in the middle of a batch.  The first round's
// commit stays exact: its read-after-write predecessors were all dropped as null, so the pre-batch V[s2] is the
// maximum of the row it reads.  After the last round every kept lane refreshes the summaries of its row s (lanes
// that share a state write identical values).
template <int A, bool SUM = false>
COBEL_DEV void td_batch_level_parallel(double* Q, uint32_t* wm, uint32_t* rm, int S, int lane, bool active,
                                       int s, int a, double r, int s2, int nt, double lr, double gamma,
                                       const uint8_t* mbits = nullptr, double* td_out = nullptr,
                                       double* V = nullptr, uint8_t* P = nullptr) {
  static_assert(!SUM || A <= 4, "row summaries hold a tie pattern of at most 4 actions");
  const double g = nt ? gamma : 0.0;
  // this lane's update on the current table: returns Q[s,a] + lr*td, sets q = Q[s,a]
  auto evaluate = [&](double& q, bool from_summary) -> double {
    double mx;
    if (SUM && from_summary) {
      q = Q[s * A + a];
      mx = V[s2];
    } else {
      double row[A];
      load_row<A>(Q + s2 * A, row);
      q = Q[s * A + a];
      if (mbits) {
        const uint32_t mb = mbits[s2];
        mx = -__longlong_as_double(0x7FF0000000000000ll);
#pragma unroll
        for (int x = 0; x < A; ++x) mx = (mb >> x & 1u) ? xmax(mx, row[x]) : mx;
      } else {
        mx = row_max<A>(row);
      }
    }
    double td = xadd(r, xmul(g, mx));
    td = xsub(td, q);
    if (td_out) *td_out = td;
    return xadd(q, xmul(lr, td));
  };
  // speculative pass against the pre-batch table; bit equality, so that -0.0 and +0.0 differ
  double qn = 0.0;
  bool null = true;                                                 // inactive lanes count as null
  if (active) {
    double q;
    qn = evaluate(q, true);
    null = __double_as_longlong(qn) == __double_as_longlong(q);
  }
  unsigned bad = __ballot_sync(kFull, !null);
  if (bad == 0) return;                                             // every update is a no-op

  const unsigned below = (1u << lane) - 1u;
  // writers / readers per state (wm / rm are all-zero on entry and are re-zeroed on exit)
  if (active) {
    // shared-memory OR reductions (fire-and-forget RED.OR) instead of two MATCH.ANY: the masks are only needed
    // after the barrier below
    atomicOr(&wm[s], 1u << lane);
    atomicOr(&rm[s2], 1u << lane);
  }
  // lanes with my action, from A cheap ballots instead of a third MATCH
  unsigned same_a = 0;
#pragma unroll
  for (int x = 0; x < A; ++x) {
    const unsigned bx = __ballot_sync(kFull, active && a == x);
    same_a = a == x ? bx : same_a;
  }
  __syncwarp();
  unsigned raw = 0, dep = 0;                                        // earlier lanes this update has to wait for
  if (active) {
    raw = (wm[s2] | (wm[s] & same_a)) & below;                      // i writes into the row / the entry j reads
    dep = raw | (rm[s] & below);                                    // j writes into the row i reads
  }
  __syncwarp();
  if (active) { wm[s] = 0; rm[s2] = 0; }
  // valid lanes: a fixpoint from "all valid"; the set only shrinks, so `bad` (= not valid-and-null) only grows
  for (;;) {
    const bool valid = (raw & bad) == 0;
    const unsigned b = __ballot_sync(kFull, !(valid && null));
    if (b == bad) break;
    bad = b;
  }
  dep &= bad;                                                       // the kept updates; dropped ones order nothing
  unsigned done = ~bad;
  for (bool first = true; done != kFull; first = false) {
    const bool ready = !(done >> lane & 1u) && (dep & ~done) == 0;
    const unsigned R = __ballot_sync(kFull, ready);
    // the lanes of a round touch disjoint data (every read-write and write-write overlap is a dependence above),
    // so a lane writes straight after its reads; one barrier per round orders the rounds
    if (ready) {
      double q;
      Q[s * A + a] = first ? qn : evaluate(q, false);
    }
    __syncwarp();
    done |= R;
  }
  if constexpr (SUM) {
    if (bad >> lane & 1u) refresh_row_summary<A>(Q, V, P, s);
    __syncwarp();
  }
}
