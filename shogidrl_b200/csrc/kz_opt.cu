// kz_opt.cu -- the tail of a PPO minibatch update on sm_100a: global gradient-norm clipping + Adam in three launches
//   (keisei/core/ppo_agent.py:405-413: clip_grad_norm_(parameters, gradient_clip_max_norm); optimizer.step() with
//    torch.optim.Adam, ppo_agent.py:66-80).
//
// Why a kernel: torch runs this as ~10 multi-tensor launches (norms, stack, clip coefficient, scale of every
// gradient, the Adam moments, bias corrections, addcdiv) that read and write the 70 MB of fp32 state several times
// -- 0.24 ms of a 2.6 ms update on B200 (profiles/ppo_update_breakdown_r1.txt).  HBM-bound: what has to move is one
// read of g for the norm, then one read of (p, g, m, v) and one write of (p, m, v): 32 B per parameter.
//   1. kz_sumsq_kernel      per-block partial sums of g^2 (fixed order inside a block)
//   2. kz_norm_kernel       one CTA adds the partials in a fixed order: total norm and the clip coefficient
//   3. kz_adam_kernel       g *= coef; [g += wd p]; m, v, p updated exactly as torch.optim.Adam (capturable) does
// Deterministic (no atomics).  The clipped gradients are not written back: nobody reads them after the step.
#include <cuda_runtime.h>
#include <stdint.h>
#include <vector>
#include "../../include/keisei_b200.h"

int kz_cuda_fail(cudaError_t e);  // kz_engine.cu: records the message for kz_last_cuda_error

namespace {

inline int fail(cudaError_t e) { return kz_cuda_fail(e); }

constexpr int GROUP = 16;              // tensors per launch (passed by value in the kernel parameters)
constexpr int THREADS = 256;
constexpr int PER_THREAD = 16;
constexpr int CHUNK = THREADS * PER_THREAD;  // elements per CTA

struct Group {
  float* p[GROUP];
  const float* g[GROUP];
  float* m[GROUP];
  float* v[GROUP];
  const float* step[GROUP];
  long long n[GROUP];
  int blk0[GROUP + 1];  // first CTA of tensor t within this launch
  int count;
  int partial0;         // index of this launch's first partial sum
};

__device__ __forceinline__ int find_tensor(const Group& G, int b) {
  int t = 0;
#pragma unroll 1
  while (t + 1 < G.count && b >= G.blk0[t + 1]) t++;
  return t;
}

__device__ __forceinline__ float block_sum(float v) {
  __shared__ float red[THREADS / 32];
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float tot = 0.f;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < THREADS / 32; i++) tot += red[i];
  }
  return tot;  // valid in thread 0
}

__global__ void __launch_bounds__(THREADS) kz_sumsq_kernel(const Group G, float* __restrict__ partials) {
  const int t = find_tensor(G, blockIdx.x);
  const long long base = (long long)(blockIdx.x - G.blk0[t]) * CHUNK;
  const long long n = G.n[t];
  const float* __restrict__ g = G.g[t];
  float acc = 0.f;
  if (base + CHUNK <= n && ((uintptr_t)g & 15) == 0) {
    const float4* g4 = reinterpret_cast<const float4*>(g + base);
#pragma unroll
    for (int k = 0; k < PER_THREAD / 4; k++) {
      const float4 x = g4[threadIdx.x + k * THREADS];
      acc += x.x * x.x + x.y * x.y + x.z * x.z + x.w * x.w;
    }
  } else {
    for (long long i = base + threadIdx.x; i < n && i < base + CHUNK; i += THREADS) acc += g[i] * g[i];
  }
  const float tot = block_sum(acc);
  if (threadIdx.x == 0) partials[G.partial0 + blockIdx.x] = tot;
}

// out2[0] = total L2 norm of all gradients, out2[1] = clip coefficient min(1, max_norm / (norm + 1e-6))
// (torch.nn.utils.clip_grad_norm_: clip_coef = max_norm / (total_norm + 1e-6), clamped to 1).  A NaN norm gives a NaN
// coefficient, as torch.clamp does (fminf would give 1: an unclipped step on every finite gradient).
__global__ void __launch_bounds__(1024) kz_norm_kernel(const float* __restrict__ partials, int count, float max_norm,
                                                       float* __restrict__ out2) {
  __shared__ float red[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < count; i += 1024) acc += partials[i];
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = red[threadIdx.x];
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    if (threadIdx.x == 0) {
      const float norm = sqrtf(v);
      out2[0] = norm;
      const float coef = max_norm / (norm + 1e-6f);
      out2[1] = coef > 1.0f ? 1.0f : coef;
    }
  }
}

struct Hyper {
  float lr, beta1, beta2, eps, weight_decay;
  float omb1, omb2;  // 1 - beta, formed in double on the host as torch does (1 - 0.999f in fp32 is off by 1.3e-5)
};

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, const Hyper& H, float coef, float step_size,
                                         float inv_bc2_sqrt) {
  g *= coef;
  if (H.weight_decay != 0.f) g = fmaf(H.weight_decay, p, g);
  m = m + (g - m) * H.omb1;                // exp_avg.lerp_(grad, 1 - beta1)
  v = H.beta2 * v + H.omb2 * (g * g);      // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
  const float denom = sqrtf(v) * inv_bc2_sqrt + H.eps;
  p -= step_size * (m / denom);
}

__global__ void __launch_bounds__(THREADS) kz_adam_kernel(const Group G, const Hyper H, const float* __restrict__ norm2) {
  const int t = find_tensor(G, blockIdx.x);
  const long long base = (long long)(blockIdx.x - G.blk0[t]) * CHUNK;
  const long long n = G.n[t];
  float* __restrict__ p = G.p[t];
  const float* __restrict__ g = G.g[t];
  float* __restrict__ m = G.m[t];
  float* __restrict__ v = G.v[t];
  const float coef = norm2[1];
  const float step = *G.step[t];  // already incremented by the caller (capturable Adam keeps it on the device)
  const float bc1 = 1.0f - powf(H.beta1, step);
  const float bc2 = 1.0f - powf(H.beta2, step);
  const float step_size = H.lr / bc1;
  const float inv_bc2_sqrt = 1.0f / sqrtf(bc2);
  const bool vec = base + CHUNK <= n &&
                   (((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0;
  if (vec) {
    float4* p4 = reinterpret_cast<float4*>(p + base);
    const float4* g4 = reinterpret_cast<const float4*>(g + base);
    float4* m4 = reinterpret_cast<float4*>(m + base);
    float4* v4 = reinterpret_cast<float4*>(v + base);
#pragma unroll
    for (int k = 0; k < PER_THREAD / 4; k++) {
      const int i = threadIdx.x + k * THREADS;
      float4 pp = p4[i], mm = m4[i], vv = v4[i];
      const float4 gg = g4[i];
      adam_one(pp.x, gg.x, mm.x, vv.x, H, coef, step_size, inv_bc2_sqrt);
      adam_one(pp.y, gg.y, mm.y, vv.y, H, coef, step_size, inv_bc2_sqrt);
      adam_one(pp.z, gg.z, mm.z, vv.z, H, coef, step_size, inv_bc2_sqrt);
      adam_one(pp.w, gg.w, mm.w, vv.w, H, coef, step_size, inv_bc2_sqrt);
      p4[i] = pp; m4[i] = mm; v4[i] = vv;
    }
  } else {
    for (long long i = base + threadIdx.x; i < n && i < base + CHUNK; i += THREADS) {
      float pp = p[i], mm = m[i], vv = v[i];
      adam_one(pp, g[i], mm, vv, H, coef, step_size, inv_bc2_sqrt);
      p[i] = pp; m[i] = mm; v[i] = vv;
    }
  }
}

inline long long blocks_of(long long n) { return (n + CHUNK - 1) / CHUNK; }

}  // namespace

extern "C" {

long long kz_adam_clip_workspace(int count, const int64_t* numel) {
  if (count <= 0 || !numel) return 0;
  long long blocks = 0;
  for (int i = 0; i < count; i++) blocks += numel[i] > 0 ? blocks_of(numel[i]) : 0;
  return blocks;
}

int kz_adam_clip_step(int count, void* const* params, const void* const* grads, void* const* exp_avg,
                      void* const* exp_avg_sq, const void* const* steps, const int64_t* numel, double lr, double beta1,
                      double beta2, double eps, double weight_decay, double max_norm, float* workspace,
                      int64_t workspace_floats, float* norm_out2, void* stream) {
  if (count <= 0 || !params || !grads || !exp_avg || !exp_avg_sq || !steps || !numel || !workspace || !norm_out2)
    return KZ_E_ARG;
  if (workspace_floats < kz_adam_clip_workspace(count, numel)) return KZ_E_ARG;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const Hyper H{(float)lr, (float)beta1, (float)beta2, (float)eps, (float)weight_decay, (float)(1.0 - beta1),
                (float)(1.0 - beta2)};
  // pass 1 builds the launch groups and runs the partial sums; pass 2 (after the norm) runs Adam on the same groups
  std::vector<Group> groups;
  int partial0 = 0;
  for (int i0 = 0; i0 < count;) {
    Group G;
    G.count = 0;
    G.partial0 = partial0;
    G.blk0[0] = 0;
    while (i0 < count && G.count < GROUP) {
      if (numel[i0] > 0) {
        if (!params[i0] || !grads[i0] || !exp_avg[i0] || !exp_avg_sq[i0] || !steps[i0]) return KZ_E_ARG;
        const int t = G.count++;
        G.p[t] = static_cast<float*>(params[i0]);
        G.g[t] = static_cast<const float*>(grads[i0]);
        G.m[t] = static_cast<float*>(exp_avg[i0]);
        G.v[t] = static_cast<float*>(exp_avg_sq[i0]);
        G.step[t] = static_cast<const float*>(steps[i0]);
        G.n[t] = numel[i0];
        G.blk0[t + 1] = G.blk0[t] + (int)blocks_of(numel[i0]);
      }
      i0++;
    }
    if (G.count > 0) {
      partial0 += G.blk0[G.count];
      groups.push_back(G);
    }
  }
  if (groups.empty()) return KZ_E_ARG;
  for (const Group& G : groups) kz_sumsq_kernel<<<G.blk0[G.count], THREADS, 0, st>>>(G, workspace);
  kz_norm_kernel<<<1, 1024, 0, st>>>(workspace, partial0, (float)max_norm, norm_out2);
  for (const Group& G : groups) kz_adam_kernel<<<G.blk0[G.count], THREADS, 0, st>>>(G, H, norm_out2);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KZ_OK : fail(e);
}

}  // extern "C"
