// rl_common.cuh - what the translation units of libmdpstep.so share: the thread-local error string behind
// rl_last_error(), CUDA error / device guards, the Philox4x32-10 counter layout of every random stream, and
// the few accessors other TUs need on the opaque context (defined in mdp_step.cu).
#ifndef RL_COMMON_CUH_
#define RL_COMMON_CUH_

#include "rl_mdp_step.h"

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

// one instance per thread for the whole library (C++17 inline variable)
inline thread_local char g_rl_err[512] = "";

inline int rl_fail(int code, const char* fmt, const char* a = "", long long b = 0, long long c = 0) {
  snprintf(g_rl_err, sizeof(g_rl_err), fmt, a, b, c);
  return code;
}

#define CUDA_TRY(expr)                                                                                  \
  do {                                                                                                  \
    cudaError_t _e = (expr);                                                                            \
    if (_e != cudaSuccess) {                                                                            \
      snprintf(g_rl_err, sizeof(g_rl_err), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),     \
               __FILE__, __LINE__);                                                                     \
      return RL_ECUDA;                                                                                  \
    }                                                                                                   \
  } while (0)

struct RlDeviceGuard {
  int prev;
  bool ok;
  explicit RlDeviceGuard(int dev) : prev(-1), ok(true) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~RlDeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// context accessors for the other translation units (mdp_step.cu owns the struct)
int rl_ctx_device_of(const RlCtx* ctx);
const RlStepSpec* rl_ctx_spec_of(const RlCtx* ctx);

// ---------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11) - counter-based, so noise needs no state and no bytes.
// counter = (global env id, step lo, step hi, stream<<16 | block), key = seed.
// ---------------------------------------------------------------------------------------------------
enum {
  RL_STREAM_COMMAND = 1, RL_STREAM_RESET_COMMAND = 2, RL_STREAM_RESET_STATE = 3, RL_STREAM_RESET_JOINTS = 4,
  RL_STREAM_PIT_RESAMPLE = 5, RL_STREAM_INTERVAL_RESET = 6, RL_STREAM_INTERVAL_PUSH = 7, RL_STREAM_OBS = 16
};

__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

struct RandState {
  unsigned long long seed, step;   // step already includes the device-side common step counter
  long long env_id_offset;
};
__device__ __forceinline__ RandState rl_rand_state(const RlRandom& rnd) {
  RandState rs;
  rs.seed = rnd.seed;
  rs.step = rnd.step + (rnd.step_counter ? *rnd.step_counter : 0ull);
  rs.env_id_offset = rnd.env_id_offset;
  return rs;
}
static __device__ __noinline__ uint4 rl_philox(const RandState r, long long env, uint32_t stream, uint32_t block) {
  const unsigned long long genv = (unsigned long long)(env + r.env_id_offset);
  uint4 ctr = make_uint4((uint32_t)genv, (uint32_t)r.step, (uint32_t)(r.step >> 32) ^ (uint32_t)(genv >> 32),
                         (stream << 16) | block);
  return philox4x32_10(ctr, make_uint2((uint32_t)r.seed, (uint32_t)(r.seed >> 32)));
}

// The same draw as rl_philox, inlined into its caller. For kernels added to a translation unit whose existing kernels
// call rl_philox: a new call site of the out-of-line copy changes how the compiler fits that copy (and the code of its
// existing callers) to its call sites.
__device__ __forceinline__ uint4 rl_philox_inline(const RandState r, long long env, uint32_t stream, uint32_t block) {
  const unsigned long long genv = (unsigned long long)(env + r.env_id_offset);
  uint4 ctr = make_uint4((uint32_t)genv, (uint32_t)r.step, (uint32_t)(r.step >> 32) ^ (uint32_t)(genv >> 32),
                         (stream << 16) | block);
  return philox4x32_10(ctr, make_uint2((uint32_t)r.seed, (uint32_t)(r.seed >> 32)));
}

__device__ __forceinline__ float ld_f(const RlField& f, long long env, int c) {
  return static_cast<const float*>(f.ptr)[env * f.env_stride + (long long)c * f.comp_stride];
}
__device__ __forceinline__ void st_f(const RlField& f, long long env, int c, float v) {
  static_cast<float*>(f.ptr)[env * f.env_stride + (long long)c * f.comp_stride] = v;
}

#endif  // RL_COMMON_CUH_
