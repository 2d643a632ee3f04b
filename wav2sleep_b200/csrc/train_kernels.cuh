// Element-wise / row-wise kernels of the training path (forward re-materialisation and backward of everything that
// is not a GEMM).  fp16 storage, fp32 math, fp64 accumulation for whole-night statistics.  Exact erf GELU and its
// derivative are used here (gradients are compared against torch autograd of the reference formulas).
//
// reference autograd being replaced: InstanceNorm1d + GELU + residual of ConvBlock1D (models/blocks.py:57-71,
// 173-186), ConvLayerNorm + GELU of DilatedConvBlock (blocks.py:115-126, utils.py:9-23), nn.LayerNorm /
// MultiheadAttention / GELU of the TransformerEncoderLayer (wav2sleep.py:286-296), CrossEntropyLoss(ignore_index=-1)
// (scripts/config/training/main.yaml:41-46), clip_grad_norm_ + AdamW (training/main.yaml:21-22, optimizer/adamw.yaml).
#pragma once
#include "common.cuh"

namespace w2s {

W2S_DEVINL float gelu_grad(float x) {  // d/dx [x Phi(x)] = Phi(x) + x phi(x)
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752f));
  const float pdf = 0.3989422804014327f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}
W2S_DEVINL void unpack8(const uint4& u, float* v) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(&u);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float2 f = unpack_h2(w[q]);
    v[2 * q] = f.x;
    v[2 * q + 1] = f.y;
  }
}
W2S_DEVINL uint4 pack8(const float* v) {
  return make_uint4(pack_h2(v[0], v[1]), pack_h2(v[2], v[3]), pack_h2(v[4], v[5]), pack_h2(v[6], v[7]));
}
// Block-wide InstanceNorm constants: the fp64 division / square root is done once per (block, channel) by the first C
// threads and shared through smem (doing it per thread made the element-wise kernels fp64-bound).
// sm: [4][128] floats = mean, rstd, m1, m2
W2S_DEVINL void block_in_consts(float* sm, const double* stats, const double* sums, int b, int C, int L, float eps) {
  if ((int)threadIdx.x < C) {
    float mean, rstd;
    in_consts(stats, b, C, threadIdx.x, L, eps, mean, rstd);
    sm[threadIdx.x] = mean;
    sm[128 + threadIdx.x] = rstd;
    if (sums != nullptr) {
      const float invL = 1.0f / (float)L;
      sm[256 + threadIdx.x] = (float)sums[((size_t)b * C + threadIdx.x) * 2] * invL;
      sm[384 + threadIdx.x] = (float)sums[((size_t)b * C + threadIdx.x) * 2 + 1] * invL;
    }
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------------------------------
// A. a = GELU(IN(y)) [ -> GELU(a + r) ]   (re-materialise an activated tensor for wgrad)
// ------------------------------------------------------------------------------------------------------------
struct EncActArgs {
  const act_t* y; const act_t* r; const double* stats; act_t* a; const uint8_t* row_mask;
  int B, L, C; float eps;
};
__global__ void __launch_bounds__(256) enc_act_fwd_kernel(const EncActArgs p) {
  const int b = blockIdx.y;
  if (p.row_mask && p.row_mask[b]) return;
  const int CH = p.C / 8;
  const int n = p.L * CH;  // < 2^31 (L <= 2^27 rows)
  // the grid stride (gridDim.x * 256) is a multiple of CH, so a thread always sees the same channel chunk
  const int c8 = (int)((blockIdx.x * blockDim.x + threadIdx.x) % CH);
  __shared__ float sm[512];
  block_in_consts(sm, p.stats, nullptr, b, p.C, p.L, p.eps);
  float mean[8], rstd[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    mean[k] = sm[c8 * 8 + k];
    rstd[k] = sm[128 + c8 * 8 + k];
  }
  for (int id = blockIdx.x * blockDim.x + threadIdx.x; id < n; id += gridDim.x * blockDim.x) {
    const size_t off = ((size_t)b * p.L) * p.C + (size_t)id * 8;
    float v[8], rr[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(p.y + off)), v);
    if (p.r) unpack8(__ldg(reinterpret_cast<const uint4*>(p.r + off)), rr);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float a = gelu_tanh((v[k] - mean[k]) * rstd[k]);
      if (p.r) a = gelu_tanh(a + rr[k]);
      v[k] = a;
    }
    *reinterpret_cast<uint4*>(p.a + off) = pack8(v);
  }
}

// ------------------------------------------------------------------------------------------------------------
// B. backward through the activation(s) of one conv layer + the two InstanceNorm-backward reductions
//    plain : dxh = da * GELU'(xh)
//    block : s = GELU(xh) + r ; ds = dout * GELU'(s) ; dr = ds ; dxh = ds * GELU'(xh)
//    sums[b,c] += (sum dxh, sum dxh*xh)
// ------------------------------------------------------------------------------------------------------------
struct EncActBwdArgs {
  const act_t* dout; const act_t* y; const act_t* r; const double* stats;
  act_t* dxh; act_t* dr; double* sums; const uint8_t* row_mask;
  int B, L, C; float eps;
  act_t* a_out;  // optional: the activated tensor itself (what enc_act_fwd would write), for the weight gradient
};
__global__ void __launch_bounds__(256) enc_act_bwd_kernel(const EncActBwdArgs p) {
  const int b = blockIdx.y;
  if (p.row_mask && p.row_mask[b]) return;
  const int CH = p.C / 8;
  // each thread keeps one channel chunk (blockDim.x % CH == 0) and strides over rows
  const int c8 = threadIdx.x % CH;
  const int rows_per_iter = blockDim.x / CH;
  __shared__ float sm[512];
  block_in_consts(sm, p.stats, nullptr, b, p.C, p.L, p.eps);
  float mean[8], rstd[8], s0[8], s1[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    mean[k] = sm[c8 * 8 + k];
    rstd[k] = sm[128 + c8 * 8 + k];
    s0[k] = s1[k] = 0.0f;
  }
  for (int l = blockIdx.x * rows_per_iter + threadIdx.x / CH; l < p.L; l += gridDim.x * rows_per_iter) {
    const size_t off = ((size_t)b * p.L + l) * p.C + c8 * 8;
    float d[8], v[8], rr[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(p.dout + off)), d);
    unpack8(__ldg(reinterpret_cast<const uint4*>(p.y + off)), v);
    if (p.r) unpack8(__ldg(reinterpret_cast<const uint4*>(p.r + off)), rr);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float xh = (v[k] - mean[k]) * rstd[k];
      float g = d[k];
      float a, da;
      gelu_tanh_both(xh, a, da);
      if (p.r) {
        float ds;
        gelu_tanh_both(a + rr[k], a, ds);
        g *= ds;
        rr[k] = g;  // dr
      }
      g *= da;
      d[k] = g;
      v[k] = a;
      s0[k] += g;
      s1[k] = fmaf(g, xh, s1[k]);
    }
    *reinterpret_cast<uint4*>(p.dxh + off) = pack8(d);
    if (p.a_out) *reinterpret_cast<uint4*>(p.a_out + off) = pack8(v);
    if (p.r) *reinterpret_cast<uint4*>(p.dr + off) = pack8(rr);
  }
  // block reduction over the threads that share a channel chunk
  __shared__ float red[256 * 16];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    red[threadIdx.x * 16 + k] = s0[k];
    red[threadIdx.x * 16 + 8 + k] = s1[k];
  }
  __syncthreads();
  if (threadIdx.x < CH * 16) {
    const int cc = threadIdx.x / 16, k = threadIdx.x % 16;
    float t = 0.0f;
    for (int j = cc; j < blockDim.x; j += CH) t += red[j * 16 + k];
    const int c = cc * 8 + (k & 7);
    atomicAdd(&p.sums[((size_t)b * p.C + c) * 2 + (k >> 3)], (double)t);
  }
}

// ------------------------------------------------------------------------------------------------------------
// C. InstanceNorm backward: dy = rstd * (dxh - mean_L(dxh) - xh * mean_L(dxh * xh)); optional 2x zero-upsampling
//    of the output rows (row 2l of a [B, 2L, C] tensor, zeros written to row 2l+1) for the transposed stride-2 conv.
// ------------------------------------------------------------------------------------------------------------
struct EncNormBwdArgs {
  const act_t* dxh; const act_t* y; const double* stats; const double* sums; act_t* dy; const uint8_t* row_mask;
  int B, L, C, upsample; float eps;
};
__global__ void __launch_bounds__(256) enc_norm_bwd_kernel(const EncNormBwdArgs p) {
  const int b = blockIdx.y;
  if (p.row_mask && p.row_mask[b]) return;
  const int CH = p.C / 8;
  const int n = p.L * CH;
  const int ch_shift = 31 - __clz(CH);  // CH is a power of two
  const float invL = 1.0f / (float)p.L;
  const int c8 = (int)((blockIdx.x * blockDim.x + threadIdx.x) % CH);  // fixed per thread (see above)
  __shared__ float sm[512];
  block_in_consts(sm, p.stats, p.sums, b, p.C, p.L, p.eps);
  (void)invL;
  float mean[8], rstd[8], m1[8], m2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int c = c8 * 8 + k;
    mean[k] = sm[c];
    rstd[k] = sm[128 + c];
    m1[k] = sm[256 + c];
    m2[k] = sm[384 + c];
  }
  for (int id = blockIdx.x * blockDim.x + threadIdx.x; id < n; id += gridDim.x * blockDim.x) {
    const size_t l = (size_t)(id >> ch_shift);
    const size_t off = ((size_t)b * p.L + l) * p.C + c8 * 8;
    float d[8], v[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(p.dxh + off)), d);
    unpack8(__ldg(reinterpret_cast<const uint4*>(p.y + off)), v);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float xh = (v[k] - mean[k]) * rstd[k];
      d[k] = rstd[k] * (d[k] - m1[k] - xh * m2[k]);
    }
    const size_t oo = p.upsample ? ((size_t)b * 2 * p.L + 2 * l) * p.C + c8 * 8 : off;
    *reinterpret_cast<uint4*>(p.dy + oo) = pack8(d);
    if (p.upsample) *reinterpret_cast<uint4*>(p.dy + oo + p.C) = make_uint4(0u, 0u, 0u, 0u);  // odd rows: zeros
  }
}

// ------------------------------------------------------------------------------------------------------------
// D. weight gradients of the Cin = 1 layers of block 0: dW1[c, t] = sum dy1[b,l,c] x[b,l+t-1],
//    dWds[c] = sum dr[b,j,c] x[b,2j]
// ------------------------------------------------------------------------------------------------------------
struct FirstWgradArgs {
  const float* x; const act_t* dy1; const act_t* dr; float* dw1; float* dwds; const uint8_t* row_mask;
  int B, T;
  float scale;  // 1 / loss scale of the incoming activation gradients
};
__global__ void __launch_bounds__(256) first_conv_wgrad_kernel(const FirstWgradArgs p) {
  const int b = blockIdx.y;
  if (p.row_mask && p.row_mask[b]) return;
  const float* xb = p.x + (size_t)b * p.T;
  float acc[64];
#pragma unroll
  for (int k = 0; k < 64; ++k) acc[k] = 0.0f;
  for (int l = blockIdx.x * blockDim.x + threadIdx.x; l < p.T; l += gridDim.x * blockDim.x) {
    float xm = l > 0 ? xb[l - 1] : 0.0f, x0 = xb[l], xp = l + 1 < p.T ? xb[l + 1] : 0.0f;
    xm = isinf(xm) ? 0.0f : xm; x0 = isinf(x0) ? 0.0f : x0; xp = isinf(xp) ? 0.0f : xp;
    float d[16];
    const uint4* dp = reinterpret_cast<const uint4*>(p.dy1 + ((size_t)b * p.T + l) * 16);
    unpack8(__ldg(dp), d);
    unpack8(__ldg(dp + 1), d + 8);
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      acc[c * 3] = fmaf(d[c], xm, acc[c * 3]);
      acc[c * 3 + 1] = fmaf(d[c], x0, acc[c * 3 + 1]);
      acc[c * 3 + 2] = fmaf(d[c], xp, acc[c * 3 + 2]);
    }
    if ((l & 1) == 0) {
      const uint4* rp = reinterpret_cast<const uint4*>(p.dr + ((size_t)b * (p.T >> 1) + (l >> 1)) * 16);
      unpack8(__ldg(rp), d);
      unpack8(__ldg(rp + 1), d + 8);
#pragma unroll
      for (int c = 0; c < 16; ++c) acc[48 + c] = fmaf(d[c], x0, acc[48 + c]);
    }
  }
  __shared__ float red[64];
  if (threadIdx.x < 64) red[threadIdx.x] = 0.0f;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 64; ++k) {
    float v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(&red[k], v);
  }
  __syncthreads();
  if (threadIdx.x < 48) atomicAdd(&p.dw1[threadIdx.x], red[threadIdx.x] * p.scale);
  else if (threadIdx.x < 64) atomicAdd(&p.dwds[threadIdx.x - 48], red[threadIdx.x] * p.scale);
}

// ------------------------------------------------------------------------------------------------------------
// E/F/G. row-wise LayerNorm over 128 features (warp per row, lane = 4 features)
//   fwd : h = LN(x) * g + b ; optional GELU ; optional (+ res -> GELU)                    [E, seq-mixer fwd]
//   bwd : given dout wrt the final output, back to dx ; dg, db accumulated                 [F, G]
//         optional residual gradient output ds (block end) and optional additive input grad
// ------------------------------------------------------------------------------------------------------------
struct RowLnArgs {
  const act_t* x;      // [rows, 128] LN input
  const act_t* res;    // [rows, 128] residual added after the activation (block end) or null
  const float* g; const float* b;
  act_t* out;          // fwd: output ; bwd: dx
  const act_t* dout;   // bwd: gradient wrt the final output
  const act_t* dadd;   // bwd: extra gradient added to dx (e.g. residual stream), may be null
  act_t* ds;           // bwd (res != null): gradient flowing to the residual branch (= dout * GELU'(s))
  float* dg; float* db;
  long long rows; int gelu; float eps;
  float gscale;        // bwd: dg / db are accumulated times gscale (1 / loss scale of dout)
};
W2S_DEVINL float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__global__ void __launch_bounds__(256) row_ln_fwd_kernel(const RowLnArgs p) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const float4 gg = __ldg(reinterpret_cast<const float4*>(p.g) + lane);
  const float4 bb = __ldg(reinterpret_cast<const float4*>(p.b) + lane);
  for (long long r = warp0; r < p.rows; r += nwarps) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p.x + r * 128) + lane);
    const float2 a = unpack_h2(u.x), c = unpack_h2(u.y);
    const float mean = warp_sum(a.x + a.y + c.x + c.y) * (1.0f / 128.0f);
    const float d0 = a.x - mean, d1 = a.y - mean, d2 = c.x - mean, d3 = c.y - mean;
    const float rstd = rsqrtf(warp_sum(d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3) * (1.0f / 128.0f) + p.eps);
    float o0 = d0 * rstd * gg.x + bb.x, o1 = d1 * rstd * gg.y + bb.y, o2 = d2 * rstd * gg.z + bb.z,
          o3 = d3 * rstd * gg.w + bb.w;
    if (p.gelu) { o0 = gelu_erf(o0); o1 = gelu_erf(o1); o2 = gelu_erf(o2); o3 = gelu_erf(o3); }
    if (p.res) {
      const uint2 ru = __ldg(reinterpret_cast<const uint2*>(p.res + r * 128) + lane);
      const float2 ra = unpack_h2(ru.x), rc = unpack_h2(ru.y);
      o0 = gelu_erf(o0 + ra.x); o1 = gelu_erf(o1 + ra.y); o2 = gelu_erf(o2 + rc.x); o3 = gelu_erf(o3 + rc.y);
    }
    uint2 w;
    w.x = pack_h2(o0, o1);
    w.y = pack_h2(o2, o3);
    *(reinterpret_cast<uint2*>(p.out + r * 128) + lane) = w;
  }
}
__global__ void __launch_bounds__(256) row_ln_bwd_kernel(const RowLnArgs p) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const float4 gg = __ldg(reinterpret_cast<const float4*>(p.g) + lane);
  const float4 bb = __ldg(reinterpret_cast<const float4*>(p.b) + lane);
  float ag[4] = {0, 0, 0, 0}, ab[4] = {0, 0, 0, 0};
  const float gv[4] = {gg.x, gg.y, gg.z, gg.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
  for (long long r = warp0; r < p.rows; r += nwarps) {
    float x[4], d[4], xh[4];
    {
      const uint2 u = __ldg(reinterpret_cast<const uint2*>(p.x + r * 128) + lane);
      const float2 a = unpack_h2(u.x), c = unpack_h2(u.y);
      x[0] = a.x; x[1] = a.y; x[2] = c.x; x[3] = c.y;
      const uint2 du = __ldg(reinterpret_cast<const uint2*>(p.dout + r * 128) + lane);
      const float2 da = unpack_h2(du.x), dc = unpack_h2(du.y);
      d[0] = da.x; d[1] = da.y; d[2] = dc.x; d[3] = dc.y;
    }
    const float mean = warp_sum(x[0] + x[1] + x[2] + x[3]) * (1.0f / 128.0f);
    float vs = 0.0f;
#pragma unroll
    for (int k = 0; k < 4; ++k) { x[k] -= mean; vs += x[k] * x[k]; }
    const float rstd = rsqrtf(warp_sum(vs) * (1.0f / 128.0f) + p.eps);
    float rr[4] = {0, 0, 0, 0};
    if (p.res) {
      const uint2 ru = __ldg(reinterpret_cast<const uint2*>(p.res + r * 128) + lane);
      const float2 ra = unpack_h2(ru.x), rc = unpack_h2(ru.y);
      rr[0] = ra.x; rr[1] = ra.y; rr[2] = rc.x; rr[3] = rc.y;
    }
    float s1 = 0.0f, s2 = 0.0f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      xh[k] = x[k] * rstd;
      const float u = xh[k] * gv[k] + bv[k];
      float g = d[k];
      if (p.res) { g *= gelu_grad((p.gelu ? gelu_erf(u) : u) + rr[k]); rr[k] = g; }  // ds = dout GELU'(s)
      if (p.gelu) g *= gelu_grad(u);
      ag[k] += g * xh[k];
      ab[k] += g;
      d[k] = g * gv[k];  // d xh
      s1 += d[k];
      s2 += d[k] * xh[k];
    }
    s1 = warp_sum(s1) * (1.0f / 128.0f);
    s2 = warp_sum(s2) * (1.0f / 128.0f);
    float o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) o[k] = rstd * (d[k] - s1 - xh[k] * s2);
    if (p.dadd) {
      const uint2 au = __ldg(reinterpret_cast<const uint2*>(p.dadd + r * 128) + lane);
      const float2 a0 = unpack_h2(au.x), a1 = unpack_h2(au.y);
      o[0] += a0.x; o[1] += a0.y; o[2] += a1.x; o[3] += a1.y;
    }
    uint2 w;
    w.x = pack_h2(o[0], o[1]);
    w.y = pack_h2(o[2], o[3]);
    *(reinterpret_cast<uint2*>(p.out + r * 128) + lane) = w;
    if (p.res && p.ds) {
      w.x = pack_h2(rr[0], rr[1]);
      w.y = pack_h2(rr[2], rr[3]);
      *(reinterpret_cast<uint2*>(p.ds + r * 128) + lane) = w;
    }
  }
  // dg / db: reduce the 8 warps of the block through shared memory, then one atomic per feature
  __shared__ float red[8][256];
  const int w = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    red[w][lane * 4 + k] = ag[k];
    red[w][128 + lane * 4 + k] = ab[k];
  }
  __syncthreads();
  if (threadIdx.x < 256) {
    float t = 0.0f;
#pragma unroll
    for (int j = 0; j < 8; ++j) t += red[j][threadIdx.x];
    if (threadIdx.x < 128) atomicAdd(&p.dg[threadIdx.x], t * p.gscale);
    else atomicAdd(&p.db[threadIdx.x - 128], t * p.gscale);
  }
}

// ------------------------------------------------------------------------------------------------------------
// I. GELU forward / backward on flat fp16 tensors (FFN hidden, encoder linear output)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gelu_fwd_kernel(const act_t* pre, act_t* out, long long n8) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float v[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(pre) + i), v);
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = gelu_erf(v[k]);
    reinterpret_cast<uint4*>(out)[i] = pack8(v);
  }
}
__global__ void __launch_bounds__(256) gelu_bwd_kernel(const act_t* pre, const act_t* dout, act_t* din, long long n8) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float v[8], d[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(pre) + i), v);
    unpack8(__ldg(reinterpret_cast<const uint4*>(dout) + i), d);
#pragma unroll
    for (int k = 0; k < 8; ++k) d[k] *= gelu_grad(v[k]);
    reinterpret_cast<uint4*>(din)[i] = pack8(d);
  }
}

// ------------------------------------------------------------------------------------------------------------
// J. column sums of a [rows, C] fp16 matrix into fp32 (bias gradients); C <= 128, C % 8 == 0, 256 % (C / 8) == 0
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) colsum_kernel(const act_t* x, float* out, long long rows, int C, int row_stride,
                                                     int row_offset, const uint8_t* row_mask,
                                                     long long rows_per_sample, float scale) {
  const int CH = C / 8;
  const int c8 = threadIdx.x % CH;
  const int rpi = blockDim.x / CH;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (threadIdx.x < rpi * CH) {
    for (long long r = blockIdx.x * (long long)rpi + threadIdx.x / CH; r < rows; r += (long long)gridDim.x * rpi) {
      if (row_mask && row_mask[r / rows_per_sample]) continue;
      float v[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(x + (r * row_stride + row_offset) * C) + c8), v);
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] += v[k];
    }
  }
  __shared__ float red[256 * 8];
#pragma unroll
  for (int k = 0; k < 8; ++k) red[threadIdx.x * 8 + k] = acc[k];
  __syncthreads();
  if (threadIdx.x < C) {
    const int cc = threadIdx.x / 8, k = threadIdx.x % 8;
    float t = 0.0f;
    for (int j = cc; j < rpi * CH; j += CH) t += red[j * 8 + k];
    atomicAdd(&out[threadIdx.x], t * scale);
  }
}

// ------------------------------------------------------------------------------------------------------------
// J0. dropout (nn.Dropout inside nn.TransformerEncoderLayer and DilatedConvBlock, training only).
//     Counter-based: the keep decision of element idx of dropout site `site` is a pure function of (seed, site, idx),
//     so the backward regenerates the mask instead of storing it.  out = keep ? x / (1 - p) : 0  (+ res).
// ------------------------------------------------------------------------------------------------------------
W2S_DEVINL bool drop_keep(unsigned long long seed, unsigned site, unsigned idx, float p) {
  unsigned long long z = seed + (((unsigned long long)site << 32) | idx) * 0x9E3779B97F4A7C15ull;  // splitmix64
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (float)(unsigned)(z >> 40) * (1.0f / 16777216.0f) >= p;
}
struct DropArgs {
  const act_t* x; const act_t* res; act_t* out; uint8_t* mask_out;
  long long n; float p; unsigned long long seed; unsigned site;
};
__global__ void __launch_bounds__(256) dropout_kernel(const DropArgs a) {
  const long long i8 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 8;
  if (i8 >= a.n) return;
  const float scale = 1.0f / (1.0f - a.p);
  if (a.mask_out) {  // test hook: dump the keep decisions
#pragma unroll
    for (int k = 0; k < 8; ++k) a.mask_out[i8 + k] = drop_keep(a.seed, a.site, (unsigned)(i8 + k), a.p) ? 1 : 0;
    return;
  }
  float v[8], r[8];
  unpack8(__ldg(reinterpret_cast<const uint4*>(a.x + i8)), v);
  if (a.res) unpack8(__ldg(reinterpret_cast<const uint4*>(a.res + i8)), r);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    v[k] = drop_keep(a.seed, a.site, (unsigned)(i8 + k), a.p) ? v[k] * scale : 0.0f;
    if (a.res) v[k] += r[k];
  }
  *reinterpret_cast<uint4*>(a.out + i8) = pack8(v);
}

// ------------------------------------------------------------------------------------------------------------
// H. per-epoch multi-head attention over D <= 5 tokens (training path: separate Q, K, V tensors [N*D, 128])
// ------------------------------------------------------------------------------------------------------------
struct AttnArgs {
  const act_t* q; const act_t* k; const act_t* v;  // [N, D, 128]
  act_t* o;                                         // fwd: attention output [N, D, 128]
  const act_t* dout;                                // bwd: gradient wrt o
  act_t* dq; act_t* dk; act_t* dv;
  const uint8_t* key_mask;                          // [N, D] 1 = masked key (may be null)
  int N, D;
  float drop_p; unsigned long long seed; unsigned site;  // dropout on the attention weights (index ((n*8+h)*D+i)*D+j)
};
template <bool BWD>
__global__ void __launch_bounds__(128) attn_kernel(const AttnArgs p) {
  // one thread per (epoch, head); D*16 values per operand in registers
  const long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (it >= (long long)p.N * 8) return;
  const int n = (int)(it >> 3), h = (int)(it & 7);
  const int D = p.D;
  float q[5][16], k[5][16], v[5][16];
  const size_t base = (size_t)n * D * 128 + h * 16;
  for (int j = 0; j < D; ++j) {
    const uint4* qp = reinterpret_cast<const uint4*>(p.q + base + (size_t)j * 128);
    const uint4* kp = reinterpret_cast<const uint4*>(p.k + base + (size_t)j * 128);
    const uint4* vp = reinterpret_cast<const uint4*>(p.v + base + (size_t)j * 128);
    unpack8(__ldg(qp), q[j]); unpack8(__ldg(qp + 1), q[j] + 8);
    unpack8(__ldg(kp), k[j]); unpack8(__ldg(kp + 1), k[j] + 8);
    unpack8(__ldg(vp), v[j]); unpack8(__ldg(vp + 1), v[j] + 8);
  }
  float P[5][5];
  for (int i = 0; i < D; ++i) {
    float mx = -INFINITY;
    for (int j = 0; j < D; ++j) {
      float d = 0.0f;
#pragma unroll
      for (int c = 0; c < 16; ++c) d = fmaf(q[i][c], k[j][c], d);
      d = (p.key_mask && p.key_mask[(size_t)n * D + j]) ? -INFINITY : d * 0.25f;
      P[i][j] = d;
      mx = fmaxf(mx, d);
    }
    float den = 0.0f;
    for (int j = 0; j < D; ++j) { P[i][j] = __expf(P[i][j] - mx); den += P[i][j]; }
    const float inv = 1.0f / den;
    for (int j = 0; j < D; ++j) P[i][j] *= inv;
  }
  float M[5][5];  // dropout multiplier of each attention weight: 0 or 1 / (1 - p)
  {
    const float keep_scale = 1.0f / (1.0f - p.drop_p);
    for (int i = 0; i < D; ++i)
      for (int j = 0; j < D; ++j)
        M[i][j] = (p.drop_p > 0.0f && !drop_keep(p.seed, p.site, (unsigned)((it * D + i) * D + j), p.drop_p)) ? 0.0f
                  : (p.drop_p > 0.0f ? keep_scale : 1.0f);
  }
  if (!BWD) {
    for (int i = 0; i < D; ++i) {
      float o[16];
#pragma unroll
      for (int c = 0; c < 16; ++c) o[c] = 0.0f;
      for (int j = 0; j < D; ++j)
#pragma unroll
        for (int c = 0; c < 16; ++c) o[c] = fmaf(P[i][j] * M[i][j], v[j][c], o[c]);
      uint4* op = reinterpret_cast<uint4*>(p.o + base + (size_t)i * 128);
      op[0] = pack8(o);
      op[1] = pack8(o + 8);
    }
  } else {
    float dq[5][16], dk[5][16], dv[5][16];
    for (int j = 0; j < D; ++j)
#pragma unroll
      for (int c = 0; c < 16; ++c) dq[j][c] = dk[j][c] = dv[j][c] = 0.0f;
    for (int i = 0; i < D; ++i) {
      float dO[16];
      const uint4* dp = reinterpret_cast<const uint4*>(p.dout + base + (size_t)i * 128);
      unpack8(__ldg(dp), dO); unpack8(__ldg(dp + 1), dO + 8);
      float dP[5], dot = 0.0f;
      for (int j = 0; j < D; ++j) {
        float d = 0.0f;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          d = fmaf(dO[c], v[j][c], d);
          dv[j][c] = fmaf(P[i][j] * M[i][j], dO[c], dv[j][c]);
        }
        d *= M[i][j];
        dP[j] = d;
        dot = fmaf(P[i][j], d, dot);
      }
      for (int j = 0; j < D; ++j) {
        const float dS = P[i][j] * (dP[j] - dot) * 0.25f;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          dq[i][c] = fmaf(dS, k[j][c], dq[i][c]);
          dk[j][c] = fmaf(dS, q[i][c], dk[j][c]);
        }
      }
    }
    for (int j = 0; j < D; ++j) {
      uint4* a = reinterpret_cast<uint4*>(p.dq + base + (size_t)j * 128);
      uint4* b = reinterpret_cast<uint4*>(p.dk + base + (size_t)j * 128);
      uint4* c = reinterpret_cast<uint4*>(p.dv + base + (size_t)j * 128);
      a[0] = pack8(dq[j]); a[1] = pack8(dq[j] + 8);
      b[0] = pack8(dk[j]); b[1] = pack8(dk[j] + 8);
      c[0] = pack8(dv[j]); c[1] = pack8(dv[j] + 8);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// K. token tensor of the training-path epoch mixer: tokens[n, 0] = cls, tokens[n, 1 + i] = z_i[n] (0 if masked)
//    and its backward (scatter to the per-signal gradients, sum over epochs for the CLS parameter)
// ------------------------------------------------------------------------------------------------------------
struct TokenArgs {
  const act_t* z[4]; const uint8_t* row_mask[4]; const float* cls;
  act_t* tokens; uint8_t* key_mask;   // [N, D, 128], [N, D]
  const act_t* dtokens; act_t* dz[4]; float* dcls;
  int N, S, n_sig;
  float cls_scale;  // bwd: dcls is accumulated times cls_scale (1 / loss scale of dtokens)
};
__global__ void __launch_bounds__(256) tokens_fwd_kernel(const TokenArgs p) {
  const int D = p.n_sig + 1;
  const long long total = (long long)p.N * D * 16;
  for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < total; id += (long long)gridDim.x * blockDim.x) {
    const int ck = (int)(id & 15);
    const long long row = id >> 4;
    const int j = (int)(row % D);
    const long long n = row / D;
    float v[8];
    bool masked = false;
    if (j == 0) {
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = __ldg(p.cls + ck * 8 + k);
    } else {
      masked = p.row_mask[j - 1] && p.row_mask[j - 1][n / p.S];
      if (masked) {
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = 0.0f;
      } else {
        unpack8(__ldg(reinterpret_cast<const uint4*>(p.z[j - 1] + n * 128) + ck), v);
      }
    }
    *(reinterpret_cast<uint4*>(p.tokens + row * 128) + ck) = pack8(v);
    if (ck == 0) p.key_mask[row] = masked ? 1 : 0;
  }
}
__global__ void __launch_bounds__(256) tokens_bwd_kernel(const TokenArgs p) {
  const int D = p.n_sig + 1;
  const long long total = (long long)p.N * D * 16;
  float cls_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  int my_ck = -1;
  for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < total; id += (long long)gridDim.x * blockDim.x) {
    const int ck = (int)(id & 15);
    const long long row = id >> 4;
    const int j = (int)(row % D);
    const long long n = row / D;
    float v[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(p.dtokens + row * 128) + ck), v);
    if (j == 0) {
      my_ck = ck;  // (gridDim*blockDim) % 16 == 0 -> a thread always sees the same chunk index
#pragma unroll
      for (int k = 0; k < 8; ++k) cls_acc[k] += v[k];
    } else if (!(p.row_mask[j - 1] && p.row_mask[j - 1][n / p.S])) {
      *(reinterpret_cast<uint4*>(p.dz[j - 1] + n * 128) + ck) = pack8(v);
    }
  }
  if (my_ck >= 0) {
#pragma unroll
    for (int k = 0; k < 8; ++k) atomicAdd(&p.dcls[my_ck * 8 + k], cls_acc[k] * p.cls_scale);
  }
}
// strided row gather / scatter: out[n] = in[n * stride + offset]  (CLS rows <-> dense [N, 128])
__global__ void __launch_bounds__(256) rows_gather_kernel(const act_t* in, act_t* out, long long n_rows, int stride,
                                                          int offset, int scatter) {
  const long long total = n_rows * 16;
  for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < total; id += (long long)gridDim.x * blockDim.x) {
    const long long n = id >> 4;
    const int ck = (int)(id & 15);
    if (!scatter) *(reinterpret_cast<uint4*>(out + n * 128) + ck) = __ldg(reinterpret_cast<const uint4*>(in + (n * stride + offset) * 128) + ck);
    else *(reinterpret_cast<uint4*>(out + (n * stride + offset) * 128) + ck) = __ldg(reinterpret_cast<const uint4*>(in + n * 128) + ck);
  }
}

// ------------------------------------------------------------------------------------------------------------
// L. classifier + cross entropy (ignore_index = -1, mean over valid rows)
// ------------------------------------------------------------------------------------------------------------
struct HeadArgs {
  const act_t* feat;      // [N, 128]
  const float* w; const float* b;  // [C, 128], [C]
  float* logits;          // [N, C]
  const long long* labels;  // [N]
  double* loss_sum; double* count;   // scalars (zeroed by caller)
  float* loss;            // scalar out
  const float* dlogits;   // [N, C] (bwd)
  act_t* dfeat;           // [N, 128]
  float* dw; float* db;
  long long N; int C; long long ignore_index;
  float dfeat_scale;      // bwd: dfeat = dfeat_scale * dlogits W (loss scaling of the fp16 activation gradients)
};
__global__ void __launch_bounds__(256) head_fwd_kernel(const HeadArgs p) {  // logits = feat W^T + b (training fwd)
  const int lane = threadIdx.x & 31;
  const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp0; r < p.N; r += nwarps) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p.feat + r * 128) + lane);
    const float2 a = unpack_h2(u.x), c = unpack_h2(u.y);
    for (int k = 0; k < p.C; ++k) {
      const float4 w = __ldg(reinterpret_cast<const float4*>(p.w + k * 128) + lane);
      const float s = warp_sum(a.x * w.x + a.y * w.y + c.x * w.z + c.y * w.w);
      if (lane == 0) p.logits[r * p.C + k] = s + __ldg(p.b + k);
    }
  }
}
__global__ void __launch_bounds__(256) ce_loss_kernel(const HeadArgs p) {  // pass 1: sum of NLL and count of valid rows
  double ls = 0.0, cnt = 0.0;
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < p.N; r += (long long)gridDim.x * blockDim.x) {
    const long long y = p.labels[r];
    if (y == p.ignore_index) continue;
    const float* lg = p.logits + r * p.C;
    float mx = lg[0];
    for (int k = 1; k < p.C; ++k) mx = fmaxf(mx, lg[k]);
    float den = 0.0f;
    for (int k = 0; k < p.C; ++k) den += __expf(lg[k] - mx);
    ls += (double)(__logf(den) + mx - lg[y]);
    cnt += 1.0;
  }
  for (int o = 16; o > 0; o >>= 1) {
    ls += __shfl_xor_sync(0xffffffffu, ls, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(p.loss_sum, ls);
    atomicAdd(p.count, cnt);
  }
}
__global__ void __launch_bounds__(256) ce_grad_kernel(const HeadArgs p, float* dlogits) {  // pass 2
  const double cnt = *p.count;
  const float inv = cnt > 0.0 ? (float)(1.0 / cnt) : 0.0f;
  if (blockIdx.x == 0 && threadIdx.x == 0) *p.loss = cnt > 0.0 ? (float)(*p.loss_sum / cnt) : 0.0f;
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < p.N; r += (long long)gridDim.x * blockDim.x) {
    const long long y = p.labels[r];
    float* d = dlogits + r * p.C;
    if (y == p.ignore_index) {
      for (int k = 0; k < p.C; ++k) d[k] = 0.0f;
      continue;
    }
    const float* lg = p.logits + r * p.C;
    float mx = lg[0];
    for (int k = 1; k < p.C; ++k) mx = fmaxf(mx, lg[k]);
    float den = 0.0f;
    for (int k = 0; k < p.C; ++k) den += __expf(lg[k] - mx);
    for (int k = 0; k < p.C; ++k) d[k] = (__expf(lg[k] - mx) / den - (k == y ? 1.0f : 0.0f)) * inv;
  }
}
__global__ void __launch_bounds__(256) head_bwd_kernel(const HeadArgs p) {
  // dfeat = dlogits W ; dW = dlogits^T feat ; db = sum dlogits.  warp per row, lane = 4 features.
  const int lane = threadIdx.x & 31;
  const long long warp0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  float aw[8][4], ab[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { ab[k] = 0.0f; aw[k][0] = aw[k][1] = aw[k][2] = aw[k][3] = 0.0f; }
  for (long long r = warp0; r < p.N; r += nwarps) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p.feat + r * 128) + lane);
    const float2 a = unpack_h2(u.x), c = unpack_h2(u.y);
    float o[4] = {0, 0, 0, 0};
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      if (k < p.C) {
        const float d = __ldg(p.dlogits + r * p.C + k);
        const float4 w = __ldg(reinterpret_cast<const float4*>(p.w + k * 128) + lane);
        o[0] = fmaf(d, w.x, o[0]); o[1] = fmaf(d, w.y, o[1]); o[2] = fmaf(d, w.z, o[2]); o[3] = fmaf(d, w.w, o[3]);
        aw[k][0] = fmaf(d, a.x, aw[k][0]); aw[k][1] = fmaf(d, a.y, aw[k][1]);
        aw[k][2] = fmaf(d, c.x, aw[k][2]); aw[k][3] = fmaf(d, c.y, aw[k][3]);
        ab[k] += d;
      }
    }
    uint2 w2;
    w2.x = pack_h2(o[0] * p.dfeat_scale, o[1] * p.dfeat_scale);
    w2.y = pack_h2(o[2] * p.dfeat_scale, o[3] * p.dfeat_scale);
    *(reinterpret_cast<uint2*>(p.dfeat + r * 128) + lane) = w2;
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    if (k < p.C) {
#pragma unroll
      for (int q = 0; q < 4; ++q) atomicAdd(&p.dw[k * 128 + lane * 4 + q], aw[k][q]);
      if (lane == 0) atomicAdd(&p.db[k], ab[k]);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// M. global-norm clipping + AdamW on flat fp32 buffers (decoupled weight decay, bias correction as torch.optim.AdamW)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sumsq_kernel(const float* g, long long n, double* out) {
  double s = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double v = g[i];
    s += v * v;
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  __shared__ double red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int j = 0; j < (int)(blockDim.x >> 5); ++j) t += red[j];
    atomicAdd(out, t);
  }
}
struct AdamWArgs {
  float* p; const float* g; float* m; float* v; long long n;
  const double* gnorm_sq;  // device scalar: sum of squares of the (already reduced) gradient, or null = no clipping
  float lr, beta1, beta2, eps, weight_decay, max_norm, grad_scale;
  float bias_c1, bias_c2;  // 1 - beta1^t, 1 - beta2^t
  float* ema; float ema_decay;  // optional EMA of the parameters (reference trainer/callbacks.py:54-66), same pass
};
__global__ void __launch_bounds__(256) adamw_kernel(const AdamWArgs a) {
  float coef = a.grad_scale;
  if (a.gnorm_sq != nullptr && a.max_norm > 0.0f) {
    const float norm = sqrtf((float)(*a.gnorm_sq)) * a.grad_scale;
    coef *= fminf(1.0f, a.max_norm / (norm + 1e-6f));  // torch.nn.utils.clip_grad_norm_
  }
  const float step_size = a.lr / a.bias_c1;
  const float inv_sqrt_c2 = rsqrtf(a.bias_c2);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.n; i += (long long)gridDim.x * blockDim.x) {
    const float g = a.g[i] * coef;
    float p = a.p[i];
    p *= 1.0f - a.lr * a.weight_decay;
    const float m = a.beta1 * a.m[i] + (1.0f - a.beta1) * g;
    const float v = a.beta2 * a.v[i] + (1.0f - a.beta2) * g * g;
    a.m[i] = m;
    a.v[i] = v;
    const float denom = sqrtf(v) * inv_sqrt_c2 + a.eps;
    p -= step_size * m / denom;
    a.p[i] = p;
    if (a.ema != nullptr) a.ema[i] = a.ema_decay * a.ema[i] + (1.0f - a.ema_decay) * p;
  }
}

}  // namespace w2s
