// Integrated gradients: the two elementwise kernels around the model passes (wav2sleep_b200/attribution.py).
//
//   path_inputs:  out[k, b, t] = x0[b, t] + alphas[k] * (x[b, t] - x0[b, t])         ([K * B, T] fp32)
//   accumulate:   attr[b, t] (=|+=) (x - x0)[b, t] * sum_k weights[k] * grads[k, b, t]
//
// A non-finite x sample is copied unchanged onto every path point, so a row whose first sample is -inf stays missing
// at every step and the raw-signal convolutions keep reading such samples as 0; its attribution is exactly 0.
// Both kernels are HBM-bound: a thread owns one (b, t) sample, reads x / x0 once and walks k, so each of the K
// planes is read or written with coalesced stores.  Indices are 64-bit (K * B * T may exceed 2^31).
#pragma once
#include "common.cuh"

namespace w2s {
namespace ig {

constexpr int kThreads = 256;

__global__ void __launch_bounds__(kThreads) path_inputs_kernel(const float* __restrict__ x, const float* __restrict__ x0,
                                                               const float* __restrict__ alphas, int K, long long n,
                                                               float* __restrict__ out) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = x[i];
    const float b = x0 ? x0[i] : 0.0f;
    const bool keep = !isfinite(v);
    const float d = v - b;
    for (int k = 0; k < K; ++k) out[(long long)k * n + i] = keep ? v : fmaf(alphas[k], d, b);
  }
}

// The running sum lives in a register and is stored as fp32 between calls, and every step adds its own term
// d * w_k * g_k in k order: splitting the steps over several calls (first = 0) gives bitwise the one-call result.
__global__ void __launch_bounds__(kThreads) accumulate_kernel(const float* __restrict__ grads, const float* __restrict__ weights,
                                                              int K, const float* __restrict__ x, const float* __restrict__ x0,
                                                              long long n, float* __restrict__ attr, int first) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = x[i];
    if (!isfinite(v)) {
      attr[i] = 0.0f;
      continue;
    }
    const float d = v - (x0 ? x0[i] : 0.0f);
    float s = first ? 0.0f : attr[i];
    for (int k = 0; k < K; ++k) s = fmaf(d * weights[k], grads[(long long)k * n + i], s);
    attr[i] = s;
  }
}

}  // namespace ig
}  // namespace w2s
