// util.cu -- error plumbing, launch counter, the checks and the carry set-up shared by the entry points, and the
// stream-contract probe.
#include "common.cuh"
#include <atomic>
#include <cstdarg>

namespace {
thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};

__global__ void draw_uniforms_kernel(uint64_t seed, int64_t agent_id_base, int64_t n_agents,
                                     int64_t first, int64_t n_draws, double* out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_agents * n_draws) return;
  const int64_t a = i / n_draws, k = i - a * n_draws;
  CobelStream s{seed, agent_id_base, nullptr, nullptr, 0};
  Rng rng;
  rng.agent = (uint64_t)(s.agent_id_base + a);
  rng.key0 = (uint32_t)seed; rng.key1 = (uint32_t)(seed >> 32);
  rng.user = nullptr; rng.user_len = 0; rng.have = false; rng.k = 0;
  out[i] = rng.at((uint64_t)(first + k));
}
__global__ void stream_next_kernel(CobelStream s, int64_t n_agents, int64_t n_draws, double* out) {
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_agents) return;
  Rng rng; rng.init(s, a);
  for (int64_t k = 0; k < n_draws; ++k) out[a * n_draws + k] = rng.next();
  s.draw_count[a] = (int64_t)rng.k;
}
__global__ void set_carry_kernel(int64_t* carry, int stride, const int32_t* state, int64_t n_agents) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_agents) return;
  carry[n * stride] = state[n];
  for (int k = 1; k < stride; ++k) carry[n * stride + k] = 0;
}
}  // namespace

int cobel_validate_common(int64_t n_agents, const CobelWorld& w, const CobelStream& s, const CobelPolicy& pol,
                          const CobelTrace& tr, int trials, int steps) {
  COBEL_REQUIRE(n_agents > 0, COBEL_EINVAL, "n_agents must be positive");
  COBEL_REQUIRE(w.n_states > 0 && w.n_actions > 0 && w.n_starts > 0, COBEL_EINVAL, "empty world");
  COBEL_REQUIRE(w.succ && w.reward && w.terminal && w.starts, COBEL_EINVAL, "world tables missing");
  COBEL_REQUIRE(s.draw_count, COBEL_EINVAL, "stream.draw_count missing");
  COBEL_REQUIRE(pol.param && pol.kind >= 0 && pol.kind <= 2, COBEL_EINVAL, "bad policy");
  COBEL_REQUIRE(trials >= 0 && steps > 0, COBEL_EINVAL, "trials must be >= 0 and steps > 0");
  COBEL_REQUIRE(tr.n_steps && tr.n_replay && (trials == 0 || (tr.trial_steps && tr.trial_reward)), COBEL_EINVAL,
                "trace.trial_steps/trial_reward/n_steps/n_replay are mandatory");
  return COBEL_OK;
}

int cobel_set_carry(int64_t* carry, int stride, const int32_t* state, int64_t n_agents, cudaStream_t st) {
  return launch_kernel(set_carry_kernel, (unsigned)((n_agents + 127) / 128), 128, 0, st, carry, stride, state, n_agents);
}

void cobel_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
}

void cobel_count_launch() { ++g_launches; }

extern "C" int cobel_abi_version(void) { return COBEL_ABI_VERSION; }

extern "C" void cobel_last_error(char* buf, size_t len) {
  if (!buf || !len) return;
  strncpy(buf, g_err, len - 1);
  buf[len - 1] = 0;
}

extern "C" int64_t cobel_launch_count(void) { return g_launches.load(); }

extern "C" int cobel_draw_uniforms(uint64_t seed, int64_t agent_id_base, int64_t n_agents, int64_t first,
                                   int64_t n_draws, double* out, void* stream) {
  COBEL_REQUIRE(n_agents > 0 && n_draws > 0 && out, COBEL_EINVAL, "bad arguments to cobel_draw_uniforms");
  const int64_t total = n_agents * n_draws;
  draw_uniforms_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      seed, agent_id_base, n_agents, first, n_draws, out);
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}

extern "C" int cobel_stream_next(const CobelStream* s, int64_t n_agents, int64_t n_draws, double* out, void* stream) {
  COBEL_REQUIRE(s && s->draw_count && n_agents > 0 && n_draws > 0 && out, COBEL_EINVAL,
                "bad arguments to cobel_stream_next");
  stream_next_kernel<<<(unsigned)((n_agents + 127) / 128), 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      *s, n_agents, n_draws, out);
  cobel_count_launch();
  COBEL_CUDA_OK(cudaGetLastError());
  return COBEL_OK;
}

extern "C" size_t cobel_sizeof(const char* name) {
  if (!name) return 0;
#define COBEL_SZ(T) if (!strcmp(name, #T)) return sizeof(T);
  COBEL_SZ(CobelWorld) COBEL_SZ(CobelStream) COBEL_SZ(CobelPolicy) COBEL_SZ(CobelTrace)
  COBEL_SZ(CobelDynaQParams) COBEL_SZ(CobelQParams) COBEL_SZ(CobelSRParams) COBEL_SZ(CobelSRCompactParams) COBEL_SZ(CobelSFMAParams) COBEL_SZ(CobelPMAParams) COBEL_SZ(CobelExperiences)
#undef COBEL_SZ
  return 0;
}
