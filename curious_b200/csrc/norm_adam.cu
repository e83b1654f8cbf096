// Normalizer statistics, clip/normalise, Adam, polyak and checksum kernels (sm_100a).
//
// Replaces (reference flowersteam/curious):
//   baselines/her/normalizer.py:64-70   update            -> cur_norm_accumulate
//   baselines/her/normalizer.py:50-61,96-118 recompute    -> cur_norm_recompute
//   baselines/her/normalizer.py:72-82   (de)normalize     -> cur_norm_apply / cur_norm_invert
//   baselines/common/mpi_adam.py:30-35  Adam              -> cur_adam_step[_graph]
//   baselines/her/ddpg.py:456-462       target update     -> cur_polyak
//   baselines/common/mpi_adam.py:42-50  check_synced      -> cur_checksum
//   baselines/her/ddpg.py:147-152       exploration noise -> cur_action_noise (device-side option)
//
// All of these are tiny, L2-resident, launch-latency-bound elementwise/reduction kernels.  The
// arithmetic uses the explicitly rounded intrinsics (__fmul_rn, __fadd_rn, ...) so the compiler
// cannot contract into FMA: results are bit-identical to NumPy float32 evaluated in the reference's
// operation order.
#include "common.cuh"

namespace cur {

// ---------------------------------------------------------------- normalizer accumulate
// v is [n, dim] row-major.  Threads are laid over (row group, column) so that consecutive
// threads read consecutive addresses; partial sums are combined in shared memory.
constexpr int ACC_THREADS = 256;

__global__ void __launch_bounds__(ACC_THREADS)
norm_accumulate_kernel(const float* __restrict__ v, int64_t n, int dim, float* __restrict__ partial,
                       int use_atomics) {
  extern __shared__ float sh[];  // 2 * ACC_THREADS
  const int groups = ACC_THREADS / dim > 0 ? ACC_THREADS / dim : 1;
  float s = 0.f, q = 0.f;
  if (dim <= ACC_THREADS) {
    const int col = threadIdx.x % dim;
    const int grp = threadIdx.x / dim;
    if (grp < groups) {
      for (int64_t r = (int64_t)blockIdx.x * groups + grp; r < n; r += (int64_t)gridDim.x * groups) {
        float x = v[r * dim + col];
        s = __fadd_rn(s, x);
        q = __fadd_rn(q, __fmul_rn(x, x));
      }
    }
    sh[threadIdx.x] = s;
    sh[ACC_THREADS + threadIdx.x] = q;
    __syncthreads();
    if (threadIdx.x < dim) {
      float ts = 0.f, tq = 0.f;
      for (int g = 0; g < groups; ++g) {
        ts = __fadd_rn(ts, sh[g * dim + threadIdx.x]);
        tq = __fadd_rn(tq, sh[ACC_THREADS + g * dim + threadIdx.x]);
      }
      if (use_atomics) {
        atomicAdd(&partial[threadIdx.x], ts);
        atomicAdd(&partial[dim + threadIdx.x], tq);
      } else {
        partial[threadIdx.x] = __fadd_rn(partial[threadIdx.x], ts);
        partial[dim + threadIdx.x] = __fadd_rn(partial[dim + threadIdx.x], tq);
      }
    }
  } else {
    // wide rows: one thread per column, block-strided over columns, rows split over blocks
    for (int col = threadIdx.x; col < dim; col += ACC_THREADS) {
      s = 0.f; q = 0.f;
      for (int64_t r = blockIdx.x; r < n; r += gridDim.x) {
        float x = v[r * dim + col];
        s = __fadd_rn(s, x);
        q = __fadd_rn(q, __fmul_rn(x, x));
      }
      if (use_atomics) {
        atomicAdd(&partial[col], s);
        atomicAdd(&partial[dim + col], q);
      } else {
        partial[col] = __fadd_rn(partial[col], s);
        partial[dim + col] = __fadd_rn(partial[dim + col], q);
      }
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) partial[2 * dim] = __fadd_rn(partial[2 * dim], (float)n);
}

__global__ void norm_recompute_kernel(float* __restrict__ running, float* __restrict__ partial, float world,
                                      float eps, int dim, float* __restrict__ mean, float* __restrict__ std) {
  // count first (every thread needs the NEW count; it is a single float)
  const float cnt = __fadd_rn(running[2 * dim], __fdiv_rn(partial[2 * dim], world));
  __syncthreads();
  for (int k = threadIdx.x; k < dim; k += blockDim.x) {
    float s = __fadd_rn(running[k], __fdiv_rn(partial[k], world));
    float q = __fadd_rn(running[dim + k], __fdiv_rn(partial[dim + k], world));
    running[k] = s;
    running[dim + k] = q;
    partial[k] = 0.f;
    partial[dim + k] = 0.f;
    float m = __fdiv_rn(s, cnt);
    float var = __fsub_rn(__fdiv_rn(q, cnt), __fmul_rn(m, m));
    mean[k] = m;
    std[k] = __fsqrt_rn(fmaxf(__fmul_rn(eps, eps), var));
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    running[2 * dim] = cnt;
    partial[2 * dim] = 0.f;
  }
}

__global__ void norm_apply_kernel(const float* __restrict__ v, int64_t total, int dim,
                                  const float* __restrict__ mean, const float* __restrict__ std, float clip,
                                  float* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int k = (int)(i % dim);
    float x = __fdiv_rn(__fsub_rn(v[i], mean[k]), std[k]);
    out[i] = fminf(fmaxf(x, -clip), clip);
  }
}

__global__ void norm_invert_kernel(const float* __restrict__ v, int64_t total, int dim,
                                   const float* __restrict__ mean, const float* __restrict__ std,
                                   float* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int k = (int)(i % dim);
    out[i] = __fadd_rn(mean[k], __fmul_rn(v[i], std[k]));
  }
}

// ---------------------------------------------------------------- Adam / polyak
template <bool kTable>
__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ theta, const float* __restrict__ grad, float* __restrict__ m,
            float* __restrict__ v, int64_t n, float neg_a, const float* __restrict__ table, int table_len,
            const int64_t* __restrict__ step_counter, float b1, float omb1, float b2, float omb2, float eps,
            float grad_div, int step_div) {
  if (kTable) {
    long long t = *step_counter / step_div;      // 1-based: already bumped for this step
    if (t < 1) t = 1;
    neg_a = table[(t <= table_len ? t : (long long)table_len) - 1];
  }
  const int64_t n4 = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float4* th4 = reinterpret_cast<float4*>(theta);
  const float4* g4 = reinterpret_cast<const float4*>(grad);
  float4* m4 = reinterpret_cast<float4*>(m);
  float4* v4 = reinterpret_cast<float4*>(v);
  const bool div = grad_div != 1.0f;
  for (int64_t i = gid; i < n4; i += stride) {
    float4 T = th4[i], G = g4[i], M = m4[i], V = v4[i];
    if (div) { G.x = __fdiv_rn(G.x, grad_div); G.y = __fdiv_rn(G.y, grad_div); G.z = __fdiv_rn(G.z, grad_div); G.w = __fdiv_rn(G.w, grad_div); }
    adam_elem(T.x, G.x, M.x, V.x, neg_a, b1, omb1, b2, omb2, eps);
    adam_elem(T.y, G.y, M.y, V.y, neg_a, b1, omb1, b2, omb2, eps);
    adam_elem(T.z, G.z, M.z, V.z, neg_a, b1, omb1, b2, omb2, eps);
    adam_elem(T.w, G.w, M.w, V.w, neg_a, b1, omb1, b2, omb2, eps);
    th4[i] = T; m4[i] = M; v4[i] = V;
  }
  for (int64_t i = (n4 << 2) + gid; i < n; i += stride) {
    float T = theta[i], G = grad[i], M = m[i], V = v[i];
    if (div) G = __fdiv_rn(G, grad_div);
    adam_elem(T, G, M, V, neg_a, b1, omb1, b2, omb2, eps);
    theta[i] = T; m[i] = M; v[i] = V;
  }
}

__global__ void __launch_bounds__(256)
polyak_kernel(float* __restrict__ target, const float* __restrict__ main_, int64_t n, float p, float omp) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    target[i] = __fadd_rn(__fmul_rn(p, target[i]), __fmul_rn(omp, main_[i]));   // ddpg.py:462
}

__global__ void __launch_bounds__(256)
checksum_kernel(const float* __restrict__ x, int64_t n, unsigned long long* out) {
  unsigned long long acc = 0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    unsigned long long b = __float_as_uint(x[i]);
    acc += (b + 0x9E3779B97F4A7C15ull) * (b | 1ull);   // order-independent mix of the bit pattern
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

static int grid_for(int64_t n, int threads, int max_waves = 4) {
  int64_t b = (n + threads - 1) / threads;
  int64_t cap = (int64_t)sm_count() * max_waves;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}


// ---------------------------------------------------------------- exploration noise (device-side option)
// One thread per (row, pair of action components): action_noise_pair (common.cuh).
__global__ void action_noise_kernel(float* __restrict__ u, int64_t n, int dimu, float max_u, double noise_eps,
                                    double random_eps, uint64_t seed, uint64_t call) {
  const int pairs = (dimu + 1) / 2;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * pairs) return;
  const int64_t r = idx / pairs;
  const int p = (int)(idx - r * pairs);
  action_noise_pair(u, r, (uint32_t)r, p, dimu, max_u, noise_eps, random_eps, seed, call);
}

// Per-row keys: row r gets exactly what a one-row call cur_action_noise(u + r * dimu, 1, ..., seed[r], call[r]) gives it
// (counter row 0), so one launch stands for a loop of one-row get_actions calls of different agents.
__global__ void action_noise_rows_kernel(float* __restrict__ u, int64_t n, int dimu, float max_u, double noise_eps,
                                         double random_eps, const uint64_t* __restrict__ seed,
                                         const uint64_t* __restrict__ call) {
  const int pairs = (dimu + 1) / 2;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * pairs) return;
  const int64_t r = idx / pairs;
  const int p = (int)(idx - r * pairs);
  action_noise_pair(u, r, 0u, p, dimu, max_u, noise_eps, random_eps, seed[r], call[r]);
}

}  // namespace cur

using namespace cur;

extern "C" int cur_norm_accumulate(void* stream, const float* v, int64_t n, int dim, float* partial) {
  CUR_REQUIRE(v && partial, "NULL argument");
  CUR_REQUIRE(dim > 0 && n >= 0, "bad shape");
  if (n == 0) return CUR_OK;
  const int groups = ACC_THREADS / dim > 0 ? ACC_THREADS / dim : 1;
  // small inputs (the store_episode case: rollout_batch_size*T = 100 rows): one CTA, deterministic
  int blocks = 1, atomics = 0;
  if (n > 4096) {
    int64_t b = (n + (int64_t)groups * 64 - 1) / ((int64_t)groups * 64);
    blocks = (int)(b < (int64_t)sm_count() * 2 ? b : (int64_t)sm_count() * 2);
    atomics = blocks > 1;
  }
  norm_accumulate_kernel<<<blocks, ACC_THREADS, 2 * ACC_THREADS * sizeof(float), (cudaStream_t)stream>>>(
      v, n, dim, partial, atomics);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_norm_recompute(void* stream, float* running, float* partial, float world, float eps,
                                  int dim, float* mean, float* std) {
  CUR_REQUIRE(running && partial && mean && std, "NULL argument");
  CUR_REQUIRE(dim > 0 && world >= 1.0f, "bad dim/world");
  norm_recompute_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(running, partial, world, eps, dim, mean, std);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_norm_apply(void* stream, const float* v, int64_t n, int dim, const float* mean,
                              const float* std, float clip, float* out) {
  CUR_REQUIRE(v && mean && std && out, "NULL argument");
  CUR_REQUIRE(dim > 0 && n >= 0, "bad shape");
  if (n == 0) return CUR_OK;
  norm_apply_kernel<<<grid_for(n * dim, 256), 256, 0, (cudaStream_t)stream>>>(v, n * dim, dim, mean, std,
                                                                             clip, out);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_norm_invert(void* stream, const float* v, int64_t n, int dim, const float* mean,
                               const float* std, float* out) {
  CUR_REQUIRE(v && mean && std && out, "NULL argument");
  CUR_REQUIRE(dim > 0 && n >= 0, "bad shape");
  if (n == 0) return CUR_OK;
  norm_invert_kernel<<<grid_for(n * dim, 256), 256, 0, (cudaStream_t)stream>>>(v, n * dim, dim, mean, std,
                                                                              out);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_adam_step(void* stream, float* theta, const float* grad, float* m, float* v, int64_t n,
                             float neg_a, double beta1, double beta2, double eps, float grad_div) {
  CUR_REQUIRE(theta && grad && m && v, "NULL argument");
  CUR_REQUIRE(n >= 0, "negative n");
  if (n == 0) return CUR_OK;
  CUR_REQUIRE(((uintptr_t)theta | (uintptr_t)grad | (uintptr_t)m | (uintptr_t)v) % 16 == 0,
              "vectors must be 16-byte aligned");
  // python-float (1 - beta) rounded to float32, as NumPy does for a python scalar times a float32 array
  const float omb1 = (float)(1.0 - beta1), omb2 = (float)(1.0 - beta2);
  adam_kernel<false><<<grid_for(n / 4 + 1, 256, 2), 256, 0, (cudaStream_t)stream>>>(
      theta, grad, m, v, n, neg_a, nullptr, 0, nullptr, (float)beta1, omb1, (float)beta2, omb2, (float)eps, grad_div, 1);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_adam_step_graph(void* stream, float* theta, const float* grad, float* m, float* v,
                                   int64_t n, const float* neg_a_table, int table_len,
                                   const int64_t* step_counter, double beta1, double beta2, double eps,
                                   float grad_div, int32_t step_div) {
  CUR_REQUIRE(theta && grad && m && v && neg_a_table && step_counter, "NULL argument");
  CUR_REQUIRE(n >= 0 && table_len > 0, "bad sizes");
  if (n == 0) return CUR_OK;
  CUR_REQUIRE(((uintptr_t)theta | (uintptr_t)grad | (uintptr_t)m | (uintptr_t)v) % 16 == 0,
              "vectors must be 16-byte aligned");
  const float omb1 = (float)(1.0 - beta1), omb2 = (float)(1.0 - beta2);
  adam_kernel<true><<<grid_for(n / 4 + 1, 256, 2), 256, 0, (cudaStream_t)stream>>>(
      theta, grad, m, v, n, 0.f, neg_a_table, table_len, step_counter, (float)beta1, omb1, (float)beta2, omb2,
      (float)eps, grad_div, step_div > 1 ? step_div : 1);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_polyak(void* stream, float* target, const float* main_, int64_t n, double polyak) {
  CUR_REQUIRE(target && main_, "NULL argument");
  CUR_REQUIRE(n >= 0, "negative n");
  if (n == 0) return CUR_OK;
  if (polyak == 0.0) {   // init_target_net_op (ddpg.py:459-460): plain copy
    CUR_CUDA_TRY(cudaMemcpyAsync(target, main_, n * sizeof(float), cudaMemcpyDeviceToDevice,
                                 (cudaStream_t)stream));
    return CUR_OK;
  }
  // TF evaluates `1. - self.polyak` in python float64, then casts the constant to float32 (ddpg.py:462)
  const float omp = (float)(1.0 - polyak);
  polyak_kernel<<<grid_for(n, 256, 2), 256, 0, (cudaStream_t)stream>>>(target, main_, n, (float)polyak, omp);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_checksum(void* stream, const float* x, int64_t n, uint64_t* out) {
  CUR_REQUIRE(x && out, "NULL argument");
  CUR_CUDA_TRY(cudaMemsetAsync(out, 0, sizeof(uint64_t), (cudaStream_t)stream));
  if (n == 0) return CUR_OK;
  checksum_kernel<<<grid_for(n, 256, 2), 256, 0, (cudaStream_t)stream>>>(x, n, (unsigned long long*)out);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_action_noise(void* stream, float* u, int64_t n, int dimu, float max_u, double noise_eps,
                                double random_eps, uint64_t seed, uint64_t call) {
  CUR_REQUIRE(u != nullptr, "NULL argument");
  CUR_REQUIRE(n >= 0 && n < (1ll << 32) && dimu > 0, "bad shape");
  CUR_REQUIRE(noise_eps >= 0.0 && random_eps >= 0.0 && random_eps <= 1.0, "bad noise parameters");
  if (n == 0) return CUR_OK;
  const int64_t threads = n * ((dimu + 1) / 2);
  action_noise_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      u, n, dimu, max_u, noise_eps, random_eps, seed, call);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_action_noise_rows(void* stream, float* u, int64_t n, int dimu, float max_u, double noise_eps,
                                     double random_eps, const uint64_t* seed, const uint64_t* call) {
  CUR_REQUIRE(u && seed && call, "NULL argument");
  CUR_REQUIRE(n >= 0 && n < (1ll << 32) && dimu > 0, "bad shape");
  CUR_REQUIRE(noise_eps >= 0.0 && random_eps >= 0.0 && random_eps <= 1.0, "bad noise parameters");
  if (n == 0) return CUR_OK;
  const int64_t threads = n * ((dimu + 1) / 2);
  action_noise_rows_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      u, n, dimu, max_u, noise_eps, random_eps, seed, call);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}
