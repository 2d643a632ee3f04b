// Backward kernels of the general fp32 path (general.cuh): training of the NON-DEFAULT model options.
//
// Same conventions as the forward kernels: fp32 storage and math, channels-last [B, L, C] tensors, PyTorch weight
// layouts, rows of masked samples (row_mask[b] != 0) skipped so that they contribute exactly zero.  Reductions over
// positions (weight / bias / norm-parameter gradients) are parallel: position tiles per block, fp32 partials reduced in
// shared memory, fp64 atomics across blocks into a caller-provided workspace, then a finalize pass to fp32.
#pragma once
#include "general.cuh"

namespace w2s {
namespace gen {

// d act(x) / dx, exact for every activation of `activate`
W2S_DEVINL float activate_grad(float x, int act) {
  switch (act) {
    case ACT_RELU: return x > 0.0f ? 1.0f : 0.0f;
    case ACT_LEAKY: return x > 0.0f ? 1.0f : 0.01f;
    case ACT_GELU: return 0.5f * (1.0f + erff(x * 0.70710678118654752f)) + x * 0.39894228040143268f * expf(-0.5f * x * x);
    case ACT_SILU: {
      const float s = 1.0f / (1.0f + expf(-x));
      return s * (1.0f + x * (1.0f - s));
    }
    default: return 1.0f;
  }
}

constexpr int kRedWarps = 8;    // warps per reduction block: one position slice each
constexpr int kRedTile = 256;   // positions per reduction block (kRedTile / kRedWarps per warp)

// ------------------------------------------------------------------------------------------------------------
// conv data gradient (gather, one thread per input element, no atomics):
//   din[b, li, ci] = sum over (lo, t) with lo * stride - pad_left + t * dil = li of dout[b, lo, co] * w[co, ci, t]
// ------------------------------------------------------------------------------------------------------------
struct ConvBwdArgs {
  const float* in; const float* w; const float* dout; float* din; double* acc; const uint8_t* row_mask;
  int B, L_in, L_out, cin, cout, taps, stride, dil, pad_left, taps_major, raw_inf_to_zero;
};
__global__ void __launch_bounds__(256) conv_dgrad_kernel(const ConvBwdArgs p) {
  const int b = blockIdx.y;
  if (p.row_mask && p.row_mask[b]) return;
  const long long total = (long long)p.L_in * p.cin;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int li = (int)(idx / p.cin), ci = (int)(idx % p.cin);
    float acc = 0.0f;
    for (int t = 0; t < p.taps; ++t) {
      const long long num = (long long)li + p.pad_left - (long long)t * p.dil;
      if (num < 0 || num % p.stride) continue;
      const long long lo = num / p.stride;
      if (lo >= p.L_out) continue;
      const float* g = p.dout + ((size_t)b * p.L_out + lo) * p.cout;
      const float* wc = p.taps_major ? p.w + (size_t)t * p.cin + ci : p.w + (size_t)ci * p.taps + t;
      const size_t ws = p.taps_major ? (size_t)p.taps * p.cin : (size_t)p.cin * p.taps;
      for (int co = 0; co < p.cout; ++co) acc = fmaf(g[co], wc[co * ws], acc);
    }
    p.din[((size_t)b * p.L_in + li) * p.cin + ci] = acc;
  }
}

// ------------------------------------------------------------------------------------------------------------
// conv weight + bias gradient, partial sums.  Weight index k = (t * cin + ci) * cout + co (co fastest: the lanes of a
// warp read consecutive dout channels).  blockIdx.x: 32 consecutive k, blockIdx.y: tiles of kRedTile positions of the
// flattened (b, lo) range; each warp takes a slice of the tile, the 8 fp32 partials are reduced in shared memory and
// added to acc[k] (fp64).  acc[K + co] collects the bias gradient (threads with t == 0 and ci == 0).
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) conv_wgrad_kernel(const ConvBwdArgs p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long K = (long long)p.taps * p.cin * p.cout;
  const long long k = blockIdx.x * 32LL + lane;
  const bool valid = k < K;
  const int co = valid ? (int)(k % p.cout) : 0;
  const int ci = valid ? (int)((k / p.cout) % p.cin) : 0;
  const int t = valid ? (int)(k / ((long long)p.cout * p.cin)) : 0;
  const bool do_bias = valid && t == 0 && ci == 0;
  const long long npos = (long long)p.B * p.L_out;
  __shared__ float sw[kRedWarps][32], sb[kRedWarps][32];
  for (long long tile = blockIdx.y; tile * kRedTile < npos; tile += gridDim.y) {
    float aw = 0.0f, ab = 0.0f;
    if (valid) {
      const long long p0 = tile * kRedTile;
      for (int j = warp; j < kRedTile; j += kRedWarps) {
        const long long pos = p0 + j;
        if (pos >= npos) break;
        const int b = (int)(pos / p.L_out), lo = (int)(pos % p.L_out);
        if (p.row_mask && p.row_mask[b]) continue;
        const float g = p.dout[(size_t)pos * p.cout + co];
        ab += g;
        const long long li = (long long)lo * p.stride - p.pad_left + (long long)t * p.dil;
        if (li < 0 || li >= p.L_in) continue;
        float a = p.in[((size_t)b * p.L_in + li) * p.cin + ci];
        if (p.raw_inf_to_zero && isinf(a)) a = 0.0f;
        aw = fmaf(g, a, aw);
      }
    }
    sw[warp][lane] = aw;
    sb[warp][lane] = ab;
    __syncthreads();
    if (warp == 0 && valid) {
      double s = 0.0, sbias = 0.0;
      for (int w = 0; w < kRedWarps; ++w) {
        s += sw[w][lane];
        sbias += sb[w][lane];
      }
      atomicAdd(&p.acc[k], s);
      if (do_bias) atomicAdd(&p.acc[K + co], sbias);
    }
    __syncthreads();
  }
}

// acc (fp64, k = (t * cin + ci) * cout + co, then cout bias sums) -> dw in the PyTorch layout, dbias
__global__ void __launch_bounds__(256) conv_wgrad_finalize_kernel(const ConvBwdArgs p, float* dw, float* dbias) {
  const long long K = (long long)p.taps * p.cin * p.cout;
  for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < K + p.cout; k += (long long)gridDim.x * blockDim.x) {
    if (k >= K) {
      if (dbias) dbias[k - K] = (float)p.acc[k];
      continue;
    }
    if (!dw) continue;
    const int co = (int)(k % p.cout), ci = (int)((k / p.cout) % p.cin), t = (int)(k / ((long long)p.cout * p.cin));
    const size_t o = p.taps_major ? (size_t)co * p.taps * p.cin + (size_t)t * p.cin + ci : ((size_t)co * p.cin + ci) * p.taps + t;
    dw[o] = (float)p.acc[k];
  }
}

// ------------------------------------------------------------------------------------------------------------
// affine_act backward.  pre = in * scale + shift + res (recomputed exactly as the forward does), dpre = dout * act'(pre);
// din = dpre * scale; dpre itself is the residual gradient.  sums (fp64, optional): per (sample, channel) - or per
// channel when per_channel - the pair (sum dpre, sum dpre * in), i.e. the shift and scale gradients.
// Grid: x = channel groups of 32, y = position tiles of kRedTile rows, z = sample.
// ------------------------------------------------------------------------------------------------------------
struct AffineActBwdArgs {
  const float* in; const float* scale; const float* shift; const float* res; const float* dout;
  float* din; float* dpre; double* sums; const uint8_t* row_mask;
  int B, L, C, act, per_channel;
};
__global__ void __launch_bounds__(256) affine_act_bwd_kernel(const AffineActBwdArgs p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.z, c = blockIdx.x * 32 + lane;
  if (p.row_mask && p.row_mask[b]) return;
  const bool valid = c < p.C;
  const size_t ci = p.per_channel ? (size_t)c : (size_t)b * p.C + c;
  const float sc = (valid && p.scale) ? p.scale[ci] : 1.0f, sh = (valid && p.shift) ? p.shift[ci] : 0.0f;
  __shared__ float s0[kRedWarps][32], s1[kRedWarps][32];
  for (long long tile = blockIdx.y; tile * kRedTile < p.L; tile += gridDim.y) {
    float a0 = 0.0f, a1 = 0.0f;
    if (valid) {
      for (int j = warp; j < kRedTile; j += kRedWarps) {
        const long long l = tile * kRedTile + j;
        if (l >= p.L) break;
        const size_t o = ((size_t)b * p.L + l) * p.C + c;
        const float x = p.in[o];
        float v = x;
        if (p.scale) v *= sc;
        if (p.shift) v += sh;
        if (p.res) v += p.res[o];
        const float g = p.dout[o] * activate_grad(v, p.act);
        if (p.dpre) p.dpre[o] = g;
        if (p.din) p.din[o] = g * sc;
        a0 += g;
        a1 = fmaf(g, x, a1);
      }
    }
    if (p.sums) {
      s0[warp][lane] = a0;
      s1[warp][lane] = a1;
      __syncthreads();
      if (warp == 0 && valid) {
        double t0 = 0.0, t1 = 0.0;
        for (int w = 0; w < kRedWarps; ++w) {
          t0 += s0[w][lane];
          t1 += s1[w][lane];
        }
        atomicAdd(&p.sums[ci * 2], t0);
        atomicAdd(&p.sums[ci * 2 + 1], t1);
      }
      __syncthreads();
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// InstanceNorm / GroupNorm backward, coefficients.  The forward is y = x * scale + shift with scale = w * rstd,
// shift = bias - mean * w * rstd (norm_consts_kernel), so with A = sum dpre * x, S = sum dpre per (b, c) (affine_act
// backward sums) the chain rule through (mean, var) of each statistics group gives
//   dx = alpha * dpre + beta * x + gamma,   alpha = scale,  beta = 2 dvar / n,  gamma = dmean / n - 2 dvar mean / n
//   dvar = -rstd^3 / 2 * sum_c w_c (A_c - mean S_c),  dmean = -rstd * sum_c w_c S_c  (sums over the group's channels)
//   dweight[c] = sum_b rstd (A - mean S),  dbias[c] = sum_b S.
// One thread per channel, looping over the samples (B * C * channels-per-group work).  coef: [B, C, 3].
// ------------------------------------------------------------------------------------------------------------
struct NormBwdArgs {
  const double* stats; const double* sums; const float* weight; const uint8_t* row_mask;
  float* coef; float* dweight; float* dbias;
  int B, C, L, groups; float eps;
};
__global__ void __launch_bounds__(256) norm_bwd_coef_kernel(const NormBwdArgs p) {
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < p.C; c += gridDim.x * blockDim.x) {
    const int cpg = p.C / p.groups, g0 = (c / cpg) * cpg;
    const double n = (double)p.L * cpg;
    double dw = 0.0, db = 0.0;
    for (int b = 0; b < p.B; ++b) {
      if (p.row_mask && p.row_mask[b]) continue;
      double m0 = 0.0, m1 = 0.0, sa = 0.0, ss = 0.0;
      for (int k = 0; k < cpg; ++k) {
        const size_t i = (size_t)b * p.C + g0 + k;
        m0 += p.stats[i * 2];
        m1 += p.stats[i * 2 + 1];
      }
      const double mean = m0 / n, var = fmax(m1 / n - mean * mean, 0.0), rstd = 1.0 / sqrt(var + (double)p.eps);
      for (int k = 0; k < cpg; ++k) {
        const size_t i = (size_t)b * p.C + g0 + k;
        const double wk = p.weight ? (double)p.weight[g0 + k] : 1.0;
        sa += wk * (p.sums[i * 2 + 1] - mean * p.sums[i * 2]);
        ss += wk * p.sums[i * 2];
      }
      const double dvar = -0.5 * rstd * rstd * rstd * sa, dmean = -rstd * ss;
      const double wc = p.weight ? (double)p.weight[c] : 1.0;
      const size_t i = (size_t)b * p.C + c;
      p.coef[i * 3] = (float)(wc * rstd);
      p.coef[i * 3 + 1] = (float)(2.0 * dvar / n);
      p.coef[i * 3 + 2] = (float)(dmean / n - 2.0 * dvar * mean / n);
      dw += rstd * (p.sums[i * 2 + 1] - mean * p.sums[i * 2]);
      db += p.sums[i * 2];
    }
    if (p.dweight) p.dweight[c] = (float)dw;
    if (p.dbias) p.dbias[c] = (float)db;
  }
}
// dx[b, l, c] = alpha * dpre + beta * x + gamma
__global__ void __launch_bounds__(256) norm_bwd_apply_kernel(const float* x, const float* dpre, const float* coef, float* dx,
                                                             const uint8_t* row_mask, int L, int C) {
  const int b = blockIdx.y;
  if (row_mask && row_mask[b]) return;
  const long long total = (long long)L * C;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % C);
    const size_t o = (size_t)b * total + idx;
    const float* k = coef + ((size_t)b * C + c) * 3;
    dx[o] = fmaf(k[0], dpre[o], fmaf(k[1], x[o], k[2]));
  }
}

// ------------------------------------------------------------------------------------------------------------
// rownorm backward (warp per row, any C): recompute mean / rstd as the forward does, dpre = dout * act'(pre),
// g = dpre * w;  LayerNorm: dx = rstd (g - mean(g) - xhat mean(g xhat));  RMSNorm: dx = rstd (g - xhat mean(g xhat)).
// dweight / dbias: column sums of dpre * xhat / dpre, fp64 in shared memory per block, then fp64 atomics into
// acc[2 * C] (finalized by rownorm_bwd_finalize_kernel).  Dynamic shared memory: 2 * C doubles.
// ------------------------------------------------------------------------------------------------------------
struct RowNormBwdArgs {
  const float* x; const float* weight; const float* bias; const float* dout; float* dx; double* acc;
  long long rows; int C, rms, act; float eps;
};
__global__ void __launch_bounds__(256) rownorm_bwd_kernel(const RowNormBwdArgs p) {
  extern __shared__ double col[];  // [2][C]
  for (int c = threadIdx.x; c < 2 * p.C; c += blockDim.x) col[c] = 0.0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp0; r < p.rows; r += nwarps) {
    const float* row = p.x + r * p.C;
    const float* go = p.dout + r * p.C;
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
    float sg = 0.0f, sgx = 0.0f;
    for (int c = lane; c < p.C; c += 32) {
      const float xh = (row[c] - mean) * rstd;
      const float w = p.weight ? p.weight[c] : 1.0f;
      const float v = xh * w + (p.bias ? p.bias[c] : 0.0f);
      const float dp = go[c] * activate_grad(v, p.act);
      const float g = dp * w;
      sg += g;
      sgx = fmaf(g, xh, sgx);
      atomicAdd(&col[c], (double)(dp * xh));
      atomicAdd(&col[p.C + c], (double)dp);
    }
    for (int o = 16; o > 0; o >>= 1) {
      sg += __shfl_xor_sync(0xffffffffu, sg, o);
      sgx += __shfl_xor_sync(0xffffffffu, sgx, o);
    }
    const float mg = p.rms ? 0.0f : sg / (float)p.C, mgx = sgx / (float)p.C;
    for (int c = lane; c < p.C; c += 32) {
      const float xh = (row[c] - mean) * rstd;
      const float w = p.weight ? p.weight[c] : 1.0f;
      const float v = xh * w + (p.bias ? p.bias[c] : 0.0f);
      const float g = go[c] * activate_grad(v, p.act) * w;
      p.dx[r * p.C + c] = rstd * (g - mg - xh * mgx);
    }
  }
  __syncthreads();
  if (p.acc)
    for (int c = threadIdx.x; c < 2 * p.C; c += blockDim.x) atomicAdd(&p.acc[c], col[c]);
}
__global__ void __launch_bounds__(256) rownorm_bwd_finalize_kernel(const double* acc, float* dweight, float* dbias, int C) {
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
    if (dweight) dweight[c] = (float)acc[c];
    if (dbias) dbias[c] = (float)acc[C + c];
  }
}

// ------------------------------------------------------------------------------------------------------------
// attention backward (pairs with attn_kernel; same key mask, same dropout decisions).  A = softmax(q k^T * scale) over
// the unmasked keys, M = keep / (1 - p) or 0, o_i = sum_j A_ij M_ij v_j.  With dA_ij = M_ij (do_i . v_j) and
// dS_ij = A_ij (dA_ij - sum_k A_ik dA_ik):  dq_i = scale sum_j dS_ij k_j,  dk_j = scale sum_i dS_ij q_i,
// dv_j = sum_i A_ij M_ij do_i.  One thread per (epoch, head, token) computes dq of that token as a query and dk / dv of
// it as a key (re-deriving the softmax rows it needs; D is a handful of tokens), so no atomics.
// ------------------------------------------------------------------------------------------------------------
struct AttnBwdArgs {
  const float* q; const float* k; const float* v; const float* dout; float* dq; float* dk; float* dv;
  const uint8_t* key_mask;
  int N, D, H, hd, ld; float drop_p; unsigned long long seed; unsigned site;
};
W2S_DEVINL float attn_mult(const AttnBwdArgs& p, long long n, int h, int i, int j) {
  if (p.drop_p <= 0.0f) return 1.0f;
  return drop_keep(p.seed, p.site, (unsigned)(((n * p.H + h) * p.D + i) * p.D + j), p.drop_p) ? 1.0f / (1.0f - p.drop_p) : 0.0f;
}
W2S_DEVINL float attn_dot(const float* a, const float* b, int hd) {
  float d = 0.0f;
  for (int c = 0; c < hd; ++c) d = fmaf(a[c], b[c], d);
  return d;
}
// row i of epoch n, head h: max logit, softmax denominator, and sum_k A_ik dA_ik
W2S_DEVINL void attn_row(const AttnBwdArgs& p, long long n, int h, int i, float scale, float& mx, float& den, float& rd) {
  const float* qi = p.q + ((size_t)n * p.D + i) * p.ld + h * p.hd;
  const float* gi = p.dout + ((size_t)n * p.D + i) * (size_t)p.H * p.hd + h * p.hd;
  mx = -INFINITY;
  for (int j = 0; j < p.D; ++j) {
    if (p.key_mask && p.key_mask[(size_t)n * p.D + j]) continue;
    mx = fmaxf(mx, attn_dot(qi, p.k + ((size_t)n * p.D + j) * p.ld + h * p.hd, p.hd) * scale);
  }
  den = 0.0f;
  rd = 0.0f;
  for (int j = 0; j < p.D; ++j) {
    if (p.key_mask && p.key_mask[(size_t)n * p.D + j]) continue;
    const float e = expf(attn_dot(qi, p.k + ((size_t)n * p.D + j) * p.ld + h * p.hd, p.hd) * scale - mx);
    den += e;
    rd = fmaf(e, attn_mult(p, n, h, i, j) * attn_dot(gi, p.v + ((size_t)n * p.D + j) * p.ld + h * p.hd, p.hd), rd);
  }
  rd /= den;
}
__global__ void __launch_bounds__(128) attn_bwd_kernel(const AttnBwdArgs p) {
  const long long total = (long long)p.N * p.H * p.D;
  const float scale = rsqrtf((float)p.hd);
  const int F = p.H * p.hd;
  for (long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x; it < total; it += (long long)gridDim.x * blockDim.x) {
    const int t = (int)(it % p.D);
    const int h = (int)((it / p.D) % p.H);
    const long long n = it / ((long long)p.D * p.H);
    const size_t rt = (size_t)n * p.D + t;
    float* dq = p.dq + rt * p.ld + h * p.hd;
    float* dk = p.dk + rt * p.ld + h * p.hd;
    float* dv = p.dv + rt * p.ld + h * p.hd;
    for (int c = 0; c < p.hd; ++c) { dq[c] = 0.0f; dk[c] = 0.0f; dv[c] = 0.0f; }
    const float* qt = p.q + rt * p.ld + h * p.hd;
    const float* kt = p.k + rt * p.ld + h * p.hd;
    const float* vt = p.v + rt * p.ld + h * p.hd;
    // token t as the query: dq_t
    float mx, den, rd;
    attn_row(p, n, h, t, scale, mx, den, rd);
    const float* gt = p.dout + rt * F + h * p.hd;
    for (int j = 0; j < p.D; ++j) {
      if (p.key_mask && p.key_mask[(size_t)n * p.D + j]) continue;
      const float* kj = p.k + ((size_t)n * p.D + j) * p.ld + h * p.hd;
      const float a = expf(attn_dot(qt, kj, p.hd) * scale - mx) / den;
      const float da = attn_mult(p, n, h, t, j) * attn_dot(gt, p.v + ((size_t)n * p.D + j) * p.ld + h * p.hd, p.hd);
      const float ds = a * (da - rd) * scale;
      for (int c = 0; c < p.hd; ++c) dq[c] = fmaf(ds, kj[c], dq[c]);
    }
    // token t as a key: dk_t, dv_t (zero for a masked key)
    if (p.key_mask && p.key_mask[rt]) continue;
    for (int i = 0; i < p.D; ++i) {
      const size_t ri = (size_t)n * p.D + i;
      const float* qi = p.q + ri * p.ld + h * p.hd;
      const float* gi = p.dout + ri * F + h * p.hd;
      float mi, di, ri_d;
      attn_row(p, n, h, i, scale, mi, di, ri_d);
      const float a = expf(attn_dot(qi, kt, p.hd) * scale - mi) / di;
      const float m = attn_mult(p, n, h, i, t);
      const float ds = a * (m * attn_dot(gi, vt, p.hd) - ri_d) * scale;
      for (int c = 0; c < p.hd; ++c) {
        dk[c] = fmaf(ds, qi[c], dk[c]);
        dv[c] = fmaf(a * m, gi[c], dv[c]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// fp32 dropout over n elements (any n): out[i] = keep(seed, site, i) ? x[i] / (1 - p) : 0; mask_out != null: only write
// the keep decisions.  Same counter-based decisions as w2s_dropout, so applying it to the gradient is the backward.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dropout_kernel(const float* x, float* out, uint8_t* mask_out, long long n, float p,
                                                      unsigned long long seed, unsigned site) {
  const float s = 1.0f / (1.0f - p);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const bool keep = drop_keep(seed, site, (unsigned)i, p);
    if (mask_out) mask_out[i] = keep ? 1 : 0;
    else out[i] = keep ? x[i] * s : 0.0f;
  }
}

// Eval-mode BatchNorm1d parameters from the gradients of its per-channel affine (scale = w rstd, shift = b - mean w rstd,
// norm_consts_kernel with NORM_BATCH_EVAL): dweight = (dscale - running_mean dshift) rstd, dbias = dshift.
__global__ void __launch_bounds__(256) bn_eval_bwd_kernel(const float* dscale, const float* dshift, const float* running_mean,
                                                          const float* running_var, float* dweight, float* dbias, int C,
                                                          float eps) {
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
    const double rstd = 1.0 / sqrt((double)running_var[c] + (double)eps);
    if (dweight) dweight[c] = (float)(((double)dscale[c] - (double)running_mean[c] * (double)dshift[c]) * rstd);
    if (dbias) dbias[c] = dshift[c];
  }
}

}  // namespace gen
}  // namespace w2s
