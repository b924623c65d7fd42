// common.cuh -- shared device helpers: exact fp64 arithmetic, the Philox stream and
// conversion-free uniform / integer draws.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/cobel_b200.h"

#define COBEL_DEV __device__ __forceinline__

// ---------------------------------------------------------------------------
// Exact arithmetic.  Integer trajectories depend on exact float equality
// (policy/greedy.py:85 `np.amax(values) == values`, memory/pma.py:251), so every
// parity-relevant +,-,*,/ is a single IEEE round-to-nearest operation in the
// reference's order.  The __d*_rn intrinsics are never contracted into DFMA
// (the library is additionally compiled with -fmad=false).
// ---------------------------------------------------------------------------
COBEL_DEV double xadd(double a, double b) { return __dadd_rn(a, b); }
COBEL_DEV double xsub(double a, double b) { return __dsub_rn(a, b); }
COBEL_DEV double xmul(double a, double b) { return __dmul_rn(a, b); }
COBEL_DEV double xdiv(double a, double b) { return __ddiv_rn(a, b); }
// np.amax / Python max on non-NaN doubles (sign of zero is irrelevant to every consumer)
COBEL_DEV double xmax(double a, double b) { return a < b ? b : a; }

// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011), same constants as oracle/philox.py.
// ---------------------------------------------------------------------------
COBEL_DEV void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                             uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

COBEL_DEV double u53(uint32_t a, uint32_t b) {
  // ((a>>5)*2^26 + (b>>6)) * 2^-53, built without int->fp64 conversions (which are slow
  // multi-instruction sequences): placing an integer m < 2^32 in the low mantissa word of a
  // double with biased exponent 0x433-e gives (2^52 + m) * 2^-e exactly; subtracting 2^(52-e)
  // leaves m * 2^-e.  hi*2^-27 and lo*2^-53 occupy disjoint bit ranges, so the sum is exact.
  const double hi = xsub(__hiloint2double(0x43300000 - (27 << 20), (int)(a >> 5)), 33554432.0);   // (a>>5) * 2^-27
  const double lo = xsub(__hiloint2double(0x43300000 - (53 << 20), (int)(b >> 6)), 0.5);          // (b>>6) * 2^-53
  return xadd(hi, lo);
}

// One agent's uniform stream, consumed in program order (SURVEY.md Appendix A.2).
struct Rng {
  uint64_t k;              // index of the next draw
  uint64_t agent;          // global agent id
  uint32_t key0, key1;
  uint32_t w2, w3;         // second half of the block of draw k (valid when k is odd and `have`)
  bool have;
  const double* user;      // optional pre-drawn stream of this agent
  int64_t user_len;

  COBEL_DEV void init(const CobelStream& s, int64_t local_agent) {
    agent = (uint64_t)(s.agent_id_base + local_agent);
    k = (uint64_t)s.draw_count[local_agent];
    key0 = (uint32_t)s.seed; key1 = (uint32_t)(s.seed >> 32);
    have = false; w2 = w3 = 0;
    user = s.user_stream ? s.user_stream + local_agent * s.user_stream_len : nullptr;
    user_len = s.user_stream_len;
  }
  COBEL_DEV double at(uint64_t kk) const {       // random access (lane-parallel generation)
    if (user) return kk < (uint64_t)user_len ? user[kk] : 0.0;
    uint32_t o[4];
    const uint64_t b = kk >> 1;
    philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), (uint32_t)agent, (uint32_t)(agent >> 32), key0, key1, o);
    return (kk & 1) ? u53(o[2], o[3]) : u53(o[0], o[1]);
  }
  COBEL_DEV double next() {
    if (user) { const double v = k < (uint64_t)user_len ? user[k] : 0.0; ++k; return v; }
    double v;
    if ((k & 1) && have) {
      v = u53(w2, w3); have = false;
    } else {
      uint32_t o[4];
      const uint64_t b = k >> 1;
      philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), (uint32_t)agent, (uint32_t)(agent >> 32), key0, key1, o);
      if (k & 1) { v = u53(o[2], o[3]); }
      else { v = u53(o[0], o[1]); w2 = o[2]; w3 = o[3]; have = true; }
    }
    ++k;
    return v;
  }
};

// Generator.integers(n) / choice(a) from one uniform: min(floor(u*n), n-1)
// Exact int -> double for 0 <= n < 2^31 without a conversion instruction.
COBEL_DEV double int_to_f64(int n) { return xsub(__hiloint2double(0x43300000, n), 4503599627370496.0); }

COBEL_DEV int draw_integer(double u, int n) {
  // floor(u*n): adding 2^52 with round-toward-minus-infinity leaves floor(x) in the low
  // mantissa word (0 <= x < 2^31); avoids the slow fp64 -> int conversion sequence.
  const double x = xmul(u, int_to_f64(n));
  const int i = __double2loint(__dadd_rd(x, 4503599627370496.0));
  return i < n - 1 ? i : n - 1;
}

// max of a row as a balanced tree (max is exact, so the association is free): two dependent
// compare+select levels for A = 4 instead of three on the serial TD-update chain
template <int A>
COBEL_DEV double row_max(const double (&v)[A]) {
  if constexpr (A == 4) {
    return xmax(xmax(v[0], v[1]), xmax(v[2], v[3]));
  } else if constexpr (A == 6) {
    return xmax(xmax(xmax(v[0], v[1]), xmax(v[2], v[3])), xmax(v[4], v[5]));
  } else if constexpr (A == 8) {
    return xmax(xmax(xmax(v[0], v[1]), xmax(v[2], v[3])), xmax(xmax(v[4], v[5]), xmax(v[6], v[7])));
  } else {
    double m = v[0];
#pragma unroll
    for (int a = 1; a < A; ++a) m = xmax(m, v[a]);
    return m;
  }
}

// np.sum over A contiguous doubles (SURVEY.md Appendix A.3): a plain loop below 8 elements; for exactly 8 NumPy's
// pairwise routine keeps 8 accumulators and combines them as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)).
template <int A>
COBEL_DEV double np_sum(const double (&x)[A]) {
  static_assert(A <= 8, "np_sum: longer rows need the blocked pairwise tree");
  if constexpr (A == 8) {
    return xadd(xadd(xadd(x[0], x[1]), xadd(x[2], x[3])), xadd(xadd(x[4], x[5]), xadd(x[6], x[7])));
  } else {
    double s = x[0];
#pragma unroll
    for (int a = 1; a < A; ++a) s = xadd(s, x[a]);
    return s;
  }
}

// ---------------------------------------------------------------------------
// Host-side plumbing shared by the entry points: errors, the action-count dispatch, kernel launches.
// ---------------------------------------------------------------------------
void cobel_set_error(const char* fmt, ...);
void cobel_count_launch();
#define COBEL_REQUIRE(cond, code, ...)                 \
  do {                                                 \
    if (!(cond)) { cobel_set_error(__VA_ARGS__); return (code); } \
  } while (0)
#define COBEL_CUDA_OK(expr)                                                        \
  do {                                                                             \
    cudaError_t e__ = (expr);                                                      \
    if (e__ != cudaSuccess) {                                                      \
      cobel_set_error("%s failed: %s", #expr, cudaGetErrorString(e__));            \
      return COBEL_ECUDA;                                                          \
    }                                                                              \
  } while (0)

// Runs CALL with `constexpr int A` = A_ for the action counts the kernels are built for.
#define COBEL_DISPATCH_A(A_, CALL)                                                                       \
  switch (A_) {                                                                                          \
    case 2: { constexpr int A = 2; CALL; } break;                                                        \
    case 3: { constexpr int A = 3; CALL; } break;                                                        \
    case 4: { constexpr int A = 4; CALL; } break;                                                        \
    case 6: { constexpr int A = 6; CALL; } break;                                                        \
    case 8: { constexpr int A = 8; CALL; } break;                                                        \
    default: cobel_set_error("unsupported number of actions %d (built for 2,3,4,6,8)", (int)(A_)); return COBEL_EUNSUPPORTED; \
  }

// Largest dynamic shared memory of one block on sm_100 (227 KB).
constexpr int kMaxSmem = 227 * 1024;

// One kernel launch: raises the kernel's dynamic shared-memory limit to `smem`, launches, counts the launch and
// reports a launch error as COBEL_ECUDA.
template <typename... Params, typename... Args>
int launch_kernel(void (*kernel)(Params...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, const Args&... args) {
  COBEL_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<grid, block, smem, st>>>(args...);
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}

// Checks shared by the fused train()/test() entry points (util.cu).
int cobel_validate_common(int64_t n_agents, const CobelWorld& w, const CobelStream& s, const CobelPolicy& pol,
                          const CobelTrace& tr, int trials, int steps);
// replay_td is recorded entry for entry with replay_idx, so it needs that buffer: checked by every train()/test() entry
// point after its other argument checks, before a zero-trial call returns (util.cu).
int cobel_validate_replay_td(const CobelTrace& tr);
// carry[n, 0] = state[n], carry[n, 1..stride) = 0: the per-agent state a stand-alone replay starts from (util.cu).
int cobel_set_carry(int64_t* carry, int stride, const int32_t* state, int64_t n_agents, cudaStream_t st);
