// General (dimension-generic) fp32 kernels for the NON-DEFAULT model options of the reference (SURVEY section 8f, N3):
// causal / chunk-causal encoders, batch / layer / rms / group norms, relu / leaky / silu activations, feature dims
// other than 128, register tokens, signal embeddings, output norm, causal sequence mixer.
//
// reference code restated here:
//   ConvLayer1D.forward incl. the causal right-trim            models/blocks.py:173-186 (causal padding :150-152)
//   get_norm / ConvLayerNorm / ConvRMSNorm / ConvGroupNorm     models/utils.py:9-59, 77-96
//   get_activation                                            models/utils.py:61-74
//   nn.TransformerEncoderLayer (any d_model / nhead / dim_ff)  models/wav2sleep.py:286-296
//
// These configurations are not the benchmarked hot path (the default model runs on the tcgen05 kernels of
// conv_stream.cuh / conv_igemm.cuh / epoch_mixer.cuh); this is a correct CUDA path for everything else the constructors
// accept: fp32 storage and math, channels-last [B, L, C] tensors, PyTorch weight layouts, one thread per output element
// or one warp per row, fp64 statistics.  No tensor cores, nothing fused beyond norm + activation (+ residual).
#pragma once
#include "common.cuh"
#include "train_kernels.cuh"  // drop_keep: the counter-based dropout decisions of w2s_dropout

namespace w2s {
namespace gen {

enum : int { ACT_LINEAR = 0, ACT_RELU = 1, ACT_LEAKY = 2, ACT_GELU = 3, ACT_SILU = 4 };
enum : int { NORM_INSTANCE = 0, NORM_GROUP = 1, NORM_BATCH_EVAL = 2 };

W2S_DEVINL float activate(float x, int act) {
  switch (act) {
    case ACT_RELU: return fmaxf(x, 0.0f);
    case ACT_LEAKY: return x > 0.0f ? x : 0.01f * x;  // nn.LeakyReLU() default slope
    case ACT_GELU: return gelu_erf(x);
    case ACT_SILU: return x / (1.0f + expf(-x));
    default: return x;
  }
}

// ------------------------------------------------------------------------------------------------------------
// conv1d / linear: out[b, lo, co] = bias[co] + sum_{t, ci} in[b, lo*stride - pad_left + t*dil, ci] * w[co, ci, t]
// (zero outside [0, L_in)).  A causal layer of the reference (padding (k-1)*dil on both sides, right side trimmed after
// the conv) is exactly pad_left = (k-1)*dil with L_out = floor((L_in - 1) / stride) + 1.  raw_inf_to_zero: the input is
// the raw signal and non-finite samples count as 0 (models/wav2sleep.py:151).  taps_major: w is [cout, taps * cin].
// ------------------------------------------------------------------------------------------------------------
struct ConvArgs {
  const float* in; const float* w; const float* bias; float* out; const uint8_t* row_mask;
  int B, L_in, L_out, cin, cout, taps, stride, dil, pad_left, taps_major, raw_inf_to_zero;
};
__global__ void __launch_bounds__(256) conv_kernel(const ConvArgs p) {
  const int b = blockIdx.y;
  if (p.row_mask && p.row_mask[b]) return;
  const long long total = (long long)p.L_out * p.cout;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int lo = (int)(idx / p.cout), co = (int)(idx % p.cout);
    float acc = p.bias ? p.bias[co] : 0.0f;
    for (int t = 0; t < p.taps; ++t) {
      const long long li = (long long)lo * p.stride - p.pad_left + (long long)t * p.dil;
      if (li < 0 || li >= p.L_in) continue;
      const float* row = p.in + ((size_t)b * p.L_in + li) * p.cin;
      const float* wr = p.taps_major ? p.w + (size_t)co * p.taps * p.cin + (size_t)t * p.cin : p.w + (size_t)co * p.cin * p.taps + t;
      const int ws = p.taps_major ? 1 : p.taps;
      for (int ci = 0; ci < p.cin; ++ci) {
        float a = row[ci];
        if (p.raw_inf_to_zero && isinf(a)) a = 0.0f;
        acc = fmaf(a, wr[(size_t)ci * ws], acc);
      }
    }
    p.out[((size_t)b * p.L_out + lo) * p.cout + co] = acc;
  }
}

// ------------------------------------------------------------------------------------------------------------
// per-(sample, channel) sum / sum of squares over L (fp64): one block per (channel, sample)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) stats_kernel(const float* x, double* stats, const uint8_t* row_mask, int L, int C) {
  const int b = blockIdx.y, c = blockIdx.x;
  if (row_mask && row_mask[b]) return;
  double s0 = 0.0, s1 = 0.0;
  for (int l = threadIdx.x; l < L; l += blockDim.x) {
    const double v = x[((size_t)b * L + l) * C + c];
    s0 += v;
    s1 += v * v;
  }
  __shared__ double r0[256], r1[256];
  r0[threadIdx.x] = s0;
  r1[threadIdx.x] = s1;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      r0[threadIdx.x] += r0[threadIdx.x + o];
      r1[threadIdx.x] += r1[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    stats[((size_t)b * C + c) * 2] = r0[0];
    stats[((size_t)b * C + c) * 2 + 1] = r1[0];
  }
}

// ------------------------------------------------------------------------------------------------------------
// train-mode BatchNorm statistics: per-channel (sum, sum of squares) over all rows of a [rows, C] tensor (fp64).
// A channels-last [B, L, C] tensor viewed as [B * L, C] is BatchNorm's statistics group.  The block reads `span` =
// (blockDim / C) whole rows per step (C > blockDim: one blockDim-wide channel chunk of one row), so thread t always
// holds channel c0 + t % C and the warps walk contiguous bytes for any C.  kBnUnroll independent loads per thread
// are in flight before they are accumulated (fp64 per thread), then the block folds its rows in shared memory and
// adds one fp64 pair per channel to `stats` (zeroed by the caller) - one atomic per (block, channel).
// The sums are shifted by K = x[0, c] (d = x - K and d * d are exact in fp64): for |mean| >> std, sum x^2 would round
// at the scale of n * mean^2 in every cross-block addition, while sum d^2 rounds at the scale of n * var.
// bn_stats_finalize_kernel turns the shifted sums back into (sum x, sum x^2) once.
// ------------------------------------------------------------------------------------------------------------
constexpr int kBnThreads = 256, kBnUnroll = 8;
__global__ void __launch_bounds__(kBnThreads) bn_stats_kernel(const float* __restrict__ x, double* __restrict__ stats,
                                                              long long rows, int C) {
  __shared__ double r0[kBnThreads], r1[kBnThreads];
  const int t = threadIdx.x;
  for (int c0 = 0; c0 < C; c0 += kBnThreads) {
    const int cw = min(C - c0, kBnThreads);   // channels of this chunk
    const int span = kBnThreads / cw;          // rows per step
    const int ty = t / cw, tx = t % cw;
    const bool active = ty < span;
    double s0 = 0.0, s1 = 0.0;
    const long long step = (long long)span * kBnUnroll;
    if (active) {
      const float k = x[c0 + tx];
      for (long long r = (long long)blockIdx.x * step + ty; r < rows; r += (long long)gridDim.x * step) {
        float v[kBnUnroll];
#pragma unroll
        for (int u = 0; u < kBnUnroll; ++u) {
          const long long ru = r + (long long)u * span;
          v[u] = ru < rows ? x[ru * C + c0 + tx] : k;
        }
#pragma unroll
        for (int u = 0; u < kBnUnroll; ++u) {
          const double d = (double)v[u] - (double)k;
          s0 += d;
          s1 = fma(d, d, s1);
        }
      }
    }
    r0[t] = s0;
    r1[t] = s1;
    __syncthreads();
    if (t < cw) {
      double a0 = 0.0, a1 = 0.0;
      for (int k = 0; k < span; ++k) {
        a0 += r0[k * cw + t];
        a1 += r1[k * cw + t];
      }
      atomicAdd(&stats[(size_t)(c0 + t) * 2], a0);
      atomicAdd(&stats[(size_t)(c0 + t) * 2 + 1], a1);
    }
    __syncthreads();
  }
}
// (sum d, sum d^2) with d = x - K  ->  (sum x, sum x^2) = (S1 + n K, S2 + 2 K S1 + n K^2)
__global__ void __launch_bounds__(256) bn_stats_finalize_kernel(const float* __restrict__ x, double* __restrict__ stats,
                                                                long long rows, int C) {
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
    const double k = x[c], n = (double)rows;
    const double s1 = stats[(size_t)c * 2], s2 = stats[(size_t)c * 2 + 1];
    stats[(size_t)c * 2] = fma(n, k, s1);
    stats[(size_t)c * 2 + 1] = fma(n * k, k, fma(2.0 * k, s1, s2));
  }
}

// ------------------------------------------------------------------------------------------------------------
// BatchNorm1d running-statistics update of one training forward (torch.nn.functional.batch_norm, training=True):
//   num_batches_tracked += 1;  f = momentum, or 1 / num_batches_tracked when momentum < 0 (momentum=None);
//   running_mean = (1 - f) running_mean + f mean,  running_var = (1 - f) running_var + f var * n / (n - 1).
// fp64 arithmetic, fp32 buffers.  One block: every thread reads the counter before thread 0 writes it back.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bn_update_running_kernel(const double* __restrict__ stats, long long n,
                                                                float* running_mean, float* running_var,
                                                                long long* num_batches_tracked, double momentum, int C) {
  const long long tracked = *num_batches_tracked + 1;
  __syncthreads();
  if (threadIdx.x == 0) *num_batches_tracked = tracked;
  const double f = momentum < 0.0 ? 1.0 / (double)tracked : momentum;
  const double inv_n = 1.0 / (double)n, unbias = (double)n / (double)(n - 1);
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const double mean = stats[(size_t)c * 2] * inv_n;
    const double var = fmax(stats[(size_t)c * 2 + 1] * inv_n - mean * mean, 0.0);
    running_mean[c] = (float)((1.0 - f) * (double)running_mean[c] + f * mean);
    running_var[c] = (float)((1.0 - f) * (double)running_var[c] + f * var * unbias);
  }
}

// ------------------------------------------------------------------------------------------------------------
// normalisation constants: scale[b, c], shift[b, c] with y = x * scale + shift
//   NORM_INSTANCE  : nn.InstanceNorm1d (biased variance over L, no affine)              utils.py:89-92
//   NORM_GROUP     : nn.GroupNorm(groups) (statistics over L x C/groups, affine w, b)   utils.py:38-58
//   NORM_BATCH_EVAL: nn.BatchNorm1d in eval mode (running statistics, affine w, b)      utils.py:81-82
// ------------------------------------------------------------------------------------------------------------
struct NormConstArgs {
  const double* stats;  // [B, C, 2] (instance / group)
  const float* weight; const float* bias;            // [C] or null
  const float* running_mean; const float* running_var;  // [C] (batch)
  float* scale; float* shift;                         // [B, C]
  int B, C, L, mode, groups; float eps;
};
__global__ void __launch_bounds__(256) norm_consts_kernel(const NormConstArgs p) {
  const int total = p.B * p.C;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int b = idx / p.C, c = idx % p.C;
    double mean, var;
    if (p.mode == NORM_BATCH_EVAL) {
      mean = p.running_mean[c];
      var = p.running_var[c];
    } else if (p.mode == NORM_INSTANCE) {
      const double s0 = p.stats[(size_t)idx * 2], s1 = p.stats[(size_t)idx * 2 + 1];
      mean = s0 / p.L;
      var = fmax(s1 / p.L - mean * mean, 0.0);
    } else {
      const int cpg = p.C / p.groups, g0 = (c / cpg) * cpg;
      double s0 = 0.0, s1 = 0.0;
      for (int k = 0; k < cpg; ++k) {
        s0 += p.stats[((size_t)b * p.C + g0 + k) * 2];
        s1 += p.stats[((size_t)b * p.C + g0 + k) * 2 + 1];
      }
      const double n = (double)p.L * cpg;
      mean = s0 / n;
      var = fmax(s1 / n - mean * mean, 0.0);
    }
    const double rstd = 1.0 / sqrt(var + (double)p.eps);
    const double w = p.weight ? (double)p.weight[c] : 1.0, bb = p.bias ? (double)p.bias[c] : 0.0;
    p.scale[idx] = (float)(rstd * w);
    p.shift[idx] = (float)(bb - mean * rstd * w);
  }
}

// ------------------------------------------------------------------------------------------------------------
// out[b, l, c] = act( in[b, l, c] * scale[b, c] + shift[b, c] + res[b, l, c] )   (scale / shift / res optional;
// per_channel: scale / shift are [C] instead of [B, C] - eval-mode batch norm, a signal embedding added to every row)
// ------------------------------------------------------------------------------------------------------------
struct AffineActArgs {
  const float* in; const float* scale; const float* shift; const float* res; float* out; const uint8_t* row_mask;
  int B, L, C, act, per_channel;
};
__global__ void __launch_bounds__(256) affine_act_kernel(const AffineActArgs p) {
  const int b = blockIdx.y;
  if (p.row_mask && p.row_mask[b]) return;
  const long long total = (long long)p.L * p.C;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % p.C);
    const size_t o = (size_t)b * total + idx;
    float v = p.in[o];
    const size_t ci = p.per_channel ? (size_t)c : (size_t)b * p.C + c;
    if (p.scale) v *= p.scale[ci];
    if (p.shift) v += p.shift[ci];
    if (p.res) v += p.res[o];
    p.out[o] = activate(v, p.act);
  }
}

// ------------------------------------------------------------------------------------------------------------
// per-row normalisation over C features (warp per row, any C): ConvLayerNorm / nn.LayerNorm (rms = 0) or ConvRMSNorm
// (rms = 1), affine weight (+ bias), then the activation.                                   utils.py:9-36
// ------------------------------------------------------------------------------------------------------------
struct RowNormArgs {
  const float* x; const float* weight; const float* bias; float* out;
  long long rows; int C, rms, act; float eps;
};
__global__ void __launch_bounds__(256) rownorm_kernel(const RowNormArgs p) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp0; r < p.rows; r += nwarps) {
    const float* row = p.x + r * p.C;
    float s = 0.0f;
    if (!p.rms) {
      for (int c = lane; c < p.C; c += 32) s += row[c];
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    }
    const float mean = p.rms ? 0.0f : s / (float)p.C;
    float q = 0.0f;
    for (int c = lane; c < p.C; c += 32) {
      const float d = row[c] - mean;
      q = fmaf(d, d, q);
    }
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = 1.0f / sqrtf(q / (float)p.C + p.eps);
    for (int c = lane; c < p.C; c += 32) {
      float v = (row[c] - mean) * rstd * (p.weight ? p.weight[c] : 1.0f) + (p.bias ? p.bias[c] : 0.0f);
      p.out[r * p.C + c] = activate(v, p.act);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// multi-head attention over the D tokens of each epoch, any head count / head dim; q, k, v: rows of ld floats
// ([N, D, ld], head h at columns h * hd ..), o: [N, D, H * hd]; key_mask [N, D] (1 = masked key).  drop_p > 0: dropout
// on the attention weights as nn.MultiheadAttention applies it in training, keep decision drop_keep(seed, site,
// ((n * H + h) * D + query) * D + key).  One thread per (epoch, head, query).
// ------------------------------------------------------------------------------------------------------------
struct AttnArgs {
  const float* q; const float* k; const float* v; float* o; const uint8_t* key_mask;
  int N, D, H, hd, ld; float drop_p; unsigned long long seed; unsigned site;
};
__global__ void __launch_bounds__(128) attn_kernel(const AttnArgs p) {
  const long long total = (long long)p.N * p.H * p.D;
  const int F = p.H * p.hd;
  const float scale = rsqrtf((float)p.hd);
  const float keep_scale = p.drop_p > 0.0f ? 1.0f / (1.0f - p.drop_p) : 1.0f;
  for (long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x; it < total; it += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(it % p.D);
    const int h = (int)((it / p.D) % p.H);
    const long long n = it / ((long long)p.D * p.H);
    const float* qi = p.q + ((size_t)n * p.D + i) * p.ld + h * p.hd;
    float mx = -INFINITY;
    for (int j = 0; j < p.D; ++j) {
      if (p.key_mask && p.key_mask[(size_t)n * p.D + j]) continue;
      const float* kj = p.k + ((size_t)n * p.D + j) * p.ld + h * p.hd;
      float d = 0.0f;
      for (int c = 0; c < p.hd; ++c) d = fmaf(qi[c], kj[c], d);
      mx = fmaxf(mx, d * scale);
    }
    float den = 0.0f;
    float* oi = p.o + ((size_t)n * p.D + i) * F + h * p.hd;
    for (int c = 0; c < p.hd; ++c) oi[c] = 0.0f;
    for (int j = 0; j < p.D; ++j) {
      if (p.key_mask && p.key_mask[(size_t)n * p.D + j]) continue;
      const float* kj = p.k + ((size_t)n * p.D + j) * p.ld + h * p.hd;
      const float* vj = p.v + ((size_t)n * p.D + j) * p.ld + h * p.hd;
      float d = 0.0f;
      for (int c = 0; c < p.hd; ++c) d = fmaf(qi[c], kj[c], d);
      const float e = expf(d * scale - mx);
      den += e;
      float ew = e;  // the softmax denominator takes every key; dropout only scales / zeroes the weighted values
      if (p.drop_p > 0.0f)
        ew = drop_keep(p.seed, p.site, (unsigned)(((n * p.H + h) * p.D + i) * p.D + j), p.drop_p) ? e * keep_scale : 0.0f;
      for (int c = 0; c < p.hd; ++c) oi[c] = fmaf(ew, vj[c], oi[c]);
    }
    const float inv = 1.0f / den;
    for (int c = 0; c < p.hd; ++c) oi[c] *= inv;
  }
}

}  // namespace gen
}  // namespace w2s
