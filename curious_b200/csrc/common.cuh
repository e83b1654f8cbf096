// Shared helpers for the curious_b200 CUDA translation units (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/curious_b200.h"

namespace cur {

extern thread_local char g_last_error[256];

inline int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  snprintf(g_last_error, sizeof(g_last_error), "%s failed at %s:%d: %s", what, file, line,
           cudaGetErrorString(e));
  return CUR_ERR_CUDA;
}

#define CUR_CUDA_TRY(expr)                                                     \
  do {                                                                         \
    cudaError_t _e = (expr);                                                   \
    if (_e != cudaSuccess) return ::cur::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define CUR_CHECK_LAUNCH() CUR_CUDA_TRY(cudaGetLastError())

inline int invalid(const char* msg) {
  snprintf(g_last_error, sizeof(g_last_error), "invalid argument: %s", msg);
  return CUR_ERR_INVALID;
}

#define CUR_REQUIRE(cond, msg) \
  do {                         \
    if (!(cond)) return ::cur::invalid(msg); \
  } while (0)

int sm_count();

__host__ __device__ inline int round_up4(int x) { return (x + 3) & ~3; }

// ---------------------------------------------------------------- Philox4x32-10 (counter based)
struct Philox {
  uint32_t x[4];
};

__host__ __device__ inline uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

__host__ __device__ inline Philox philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = mulhi32(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = mulhi32(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  Philox p;
  p.x[0] = c0; p.x[1] = c1; p.x[2] = c2; p.x[3] = c3;
  return p;
}

// uniform in (0,1) with 32-bit resolution, as float64: (x + 0.5) * 2^-32
__host__ __device__ inline double u01_from_u32(uint32_t x) {
  return ((double)x + 0.5) * (1.0 / 4294967296.0);
}

// ---------------------------------------------------------------- exploration noise (device-side option)
// ddpg.py:147-152 on the action matrix u [n, dimu] in place, with counter-based draws instead of the host's MT19937:
//   u += noise_eps * max_u * randn(*u.shape); u = clip(u, -max_u, max_u)
//   u += binomial(1, random_eps, n)[:, None] * (uniform(-max_u, max_u, (n, dimu)) - u)
// Per (row, pair of action components): x = philox(counter = (row, pair, call_lo, call_hi ^ TAG), key = seed):
// (x0, x1) -> one Box-Muller pair, (x2, x3) -> the two uniform random-action components; the row's eps-greedy draw
// comes from the block with pair = 0xFFFFFFFF.  Arithmetic in float64 like NumPy's (the float32 action array is updated
// in place by float64 operands), rounded to float32 where the reference's `+=` rounds.  Used by cur_action_noise(_rows)
// and by the noise epilogue of the action kernel (cur_ddpg_actions_rows_noisy), which must give the same bits.
constexpr uint32_t ACTION_NOISE_TAG = 0x40000000u;

// components 2p, 2p + 1 of row r of u; `ctr` is the row's counter word (its row number in the call)
__device__ __forceinline__ void action_noise_pair(float* __restrict__ u, int64_t r, uint32_t ctr, int p, int dimu,
                                                  float max_u, double noise_eps, double random_eps, uint64_t seed,
                                                  uint64_t call) {
  const uint32_t c2 = (uint32_t)call, c3 = (uint32_t)(call >> 32) ^ ACTION_NOISE_TAG;
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const Philox x = philox4x32_10(ctr, (uint32_t)p, c2, c3, k0, k1);
  const Philox b = philox4x32_10(ctr, 0xFFFFFFFFu, c2, c3, k0, k1);
  const bool explore = u01_from_u32(b.x[0]) < random_eps;                       // binomial(1, random_eps)
  const double rad = sqrt(-2.0 * log(u01_from_u32(x.x[0])));
  const double ang = 6.283185307179586 * u01_from_u32(x.x[1]);
  const double z[2] = {__dmul_rn(rad, cos(ang)), __dmul_rn(rad, sin(ang))};
  const double mu = (double)max_u;
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int k = 2 * p + e;
    if (k >= dimu) break;
    float v = u[r * dimu + k];
    v = (float)__dadd_rn((double)v, __dmul_rn(noise_eps * mu, z[e]));           // ddpg.py:148-149 (no fma contraction)
    v = fminf(fmaxf(v, -max_u), max_u);                                         // ddpg.py:150
    if (explore) {
      const double ra = __dadd_rn(-mu, __dmul_rn(mu - (-mu), u01_from_u32(x.x[2 + e])));   // _random_action, ddpg.py:114-116
      v = (float)__dadd_rn((double)v, __dsub_rn(ra, (double)v));                // ddpg.py:151
    }
    u[r * dimu + k] = v;
  }
}

// Adam on one element: unfused IEEE float32 operations in NumPy's order (mpi_adam.py:32-35)
__device__ __forceinline__ void adam_elem(float& th, float g, float& m, float& v, float neg_a, float b1,
                                          float omb1, float b2, float omb2, float eps) {
  m = __fadd_rn(__fmul_rn(b1, m), __fmul_rn(omb1, g));                 // mpi_adam.py:32
  v = __fadd_rn(__fmul_rn(b2, v), __fmul_rn(omb2, __fmul_rn(g, g)));   // mpi_adam.py:33
  float step = __fdiv_rn(__fmul_rn(neg_a, m), __fadd_rn(__fsqrt_rn(v), eps));   // mpi_adam.py:34
  th = __fadd_rn(th, step);                                            // mpi_adam.py:35
}

}  // namespace cur
