// Fused per-epoch set transformer ("EpochMixer"): CLS token + <=4 modality tokens, all layers, one launch.
// reference: MultiModalAttentionEmbedder.forward (models/wav2sleep.py:301-346) wrapping
//            nn.TransformerEncoder(TransformerEncoderLayer(d_model=128, nhead=8, dim_ff=512, GELU,
//            batch_first, norm_first=True), num_layers) with src_key_padding_mask (wav2sleep.py:286-296,342).
//
// The problem is ~20k independent sequences of <=5 tokens: no reuse across sequences except the weights
// (0.79 MB fp16 for 2 layers, L2 resident).  One CTA processes a tile of 16 epochs (16*D token rows) with
// the fp32 residual stream, the LayerNorm output and Q/K/V resident in shared memory; the 128x{384,128,512}
// projections run as warp-level mma.sync.m16n8k16 with weight fragments streamed from L2 in pre-packed
// fragment order, the 5x5 attention runs in scalar fp32.  Rows are token-major (row = token*16 + epoch) so the
// CLS rows form exactly one 16-row MMA tile: in the last layer only K/V are computed for all tokens and
// everything else (Q, attention, out-proj, FFN) for the CLS tile alone, because only CLS is returned
// (wav2sleep.py:343-345).  Missing modalities (row_mask) are zero tokens that are masked as keys; CLS is never
// masked (wav2sleep.py:334-335).
#pragma once
#include "common.cuh"

namespace w2s {

constexpr int kMixF = 128;       // feature_dim
constexpr int kMixHeads = 8;     // nhead
constexpr int kMixHd = 16;       // head dim
constexpr int kMixFF = 512;      // dim_feedforward
constexpr int kMixEp = 16;       // epochs per tile
constexpr int kMixThreads = 256;  // measured on B200: 512 threads (16 warps) give the same 395 us per 19200 epochs
constexpr int kMixWarps = kMixThreads / 32;
constexpr int kMixMaxLayers = 8;
constexpr int kMixMaxSig = 4;

struct MixerLayerW {
  const uint2* in_w;    // packed fragments of in_proj_weight [384,128]
  const uint2* out_w;   // out_proj.weight [128,128]
  const uint2* ff1_w;   // linear1.weight [512,128]
  const uint2* ff2_w;   // linear2.weight [128,512]
  const float* in_b;    // [384]
  const float* out_b;   // [128]
  const float* ff1_b;   // [512]
  const float* ff2_b;   // [128]
  const float* ln1_w;   // [128]
  const float* ln1_b;
  const float* ln2_w;
  const float* ln2_b;
};

struct MixerArgs {
  MixerLayerW layer[kMixMaxLayers];
  int n_layers;
  const act_t* z[kMixMaxSig];          // per signal (sorted by name) [B*S, 128] encoder features
  const uint8_t* row_mask[kMixMaxSig]; // per signal [B] (1 = missing)
  const float* cls;                    // [128] register_tokens[0,0,:,0]
  act_t* out;                          // [B*S, 128]
  int n_epochs;                        // B*S
  int S;                               // epochs per night
  float ln_eps;
};

constexpr int kMixLdX = kMixF + 4;      // fp32 residual stream row stride (floats)
constexpr int kMixLdA = kMixF + 8;      // fp16 operand row stride (halfs)
constexpr int kMixLdQ = 3 * kMixF + 8;  // fp16 QKV row stride
constexpr int kMixLdH = kMixFF + 8;     // fp16 FFN hidden row stride (aliases QKV)

template <int D>
constexpr size_t mixer_smem_bytes() {
  return (size_t)16 * D * (kMixLdX * 4 + kMixLdA * 2 + kMixLdH * 2) + 16 * 8;
}

W2S_DEVINL void ldmatrix_x4(uint32_t (&a)[4], const __half* ptr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3])
               : "r"(smem_u32(ptr)));
}
W2S_DEVINL void mma_16816(float (&c)[4], const uint32_t (&a)[4], const uint2 b) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b.x), "r"(b.y));
}

// C[m_tiles*16, n8-tiles nt0..nt0+ntn) = A[., KT*16] * W^T ; epi(row, col, v0, v1) gets two adjacent columns.
// n-tiles are taken two at a time (one A fragment feeds two MMAs); an odd count ends with a single one.  (Measured:
// four at a time - half the ldmatrix traffic, 220 registers, weight fragments in chunks of 4 k-tiles - is 7 % slower.)
template <int D, int KT, class Epi>
W2S_DEVINL void warp_gemm(const __half* sAop, int lda, int m_tiles, const uint2* __restrict__ Wp, int nt0, int ntn,
                          int lane, Epi epi) {
  const int lrow = (lane & 7) + ((lane >> 3) & 1) * 8;
  const int lcol = (lane >> 4) * 8;
#pragma unroll 1
  for (int nc = 0; nc < ntn; nc += 2) {
    const bool two = nc + 1 < ntn;
    float acc[D][2][4];
#pragma unroll
    for (int m = 0; m < D; ++m)
#pragma unroll
      for (int n = 0; n < 2; ++n)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[m][n][q] = 0.0f;
#pragma unroll 1
    for (int kc = 0; kc < KT; kc += 8) {
      uint2 bf[2][8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        bf[0][k] = __ldg(Wp + ((size_t)(nt0 + nc) * KT + kc + k) * 32 + lane);
        bf[1][k] = two ? __ldg(Wp + ((size_t)(nt0 + nc + 1) * KT + kc + k) * 32 + lane) : make_uint2(0u, 0u);
      }
#pragma unroll
      for (int m = 0; m < D; ++m) {
        if (m < m_tiles) {
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            uint32_t a[4];
            ldmatrix_x4(a, sAop + (size_t)(m * 16 + lrow) * lda + (kc + k) * 16 + lcol);
            mma_16816(acc[m][0], a, bf[0][k]);
            if (two) mma_16816(acc[m][1], a, bf[1][k]);
          }
        }
      }
    }
#pragma unroll
    for (int m = 0; m < D; ++m) {
      if (m < m_tiles) {
#pragma unroll
        for (int n = 0; n < 2; ++n) {
          if (n == 1 && !two) continue;
          const int row = m * 16 + (lane >> 2);
          const int col = (nt0 + nc + n) * 8 + (lane & 3) * 2;
          epi(row, col, acc[m][n][0], acc[m][n][1]);
          epi(row + 8, col, acc[m][n][2], acc[m][n][3]);
        }
      }
    }
  }
}

// LayerNorm over 128 features of rows [0, rows): fp32 residual stream -> fp16 operand.
W2S_DEVINL void mixer_layernorm(const float* sX, __half* sA, int rows, const float* __restrict__ g,
                                const float* __restrict__ bta, float eps, int warp, int lane) {
  const float4 gg = __ldg(reinterpret_cast<const float4*>(g) + lane);
  const float4 bb = __ldg(reinterpret_cast<const float4*>(bta) + lane);
  for (int r = warp; r < rows; r += kMixThreads / 32) {
    const float4 x = *reinterpret_cast<const float4*>(sX + (size_t)r * kMixLdX + lane * 4);
    float s = x.x + x.y + x.z + x.w;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s * (1.0f / kMixF);
    const float d0 = x.x - mean, d1 = x.y - mean, d2 = x.z - mean, d3 = x.w - mean;
    float v = d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const float rstd = rsqrtf(v * (1.0f / kMixF) + eps);
    uint2 o2;
    o2.x = pack_h2(d0 * rstd * gg.x + bb.x, d1 * rstd * gg.y + bb.y);
    o2.y = pack_h2(d2 * rstd * gg.z + bb.z, d3 * rstd * gg.w + bb.w);
    *reinterpret_cast<uint2*>(sA + (size_t)r * kMixLdA + lane * 4) = o2;
  }
}

// ncu source view (round 2, profiles/r02_src_epoch_mixer.txt): the exact-erf GELU of the FFN hidden layer is 54 % of the
// executed instructions (FSEL / FFMA / FADD of erff, 49 k GELUs per tile) against 10 % HMMA - yet replacing it by the
// one-ex2 form only moves the kernel from 396 to 379 us: the tile is a chain of 14 barrier-separated phases whose
// length is set by dependent latencies (stalls: wait 26 %, short scoreboard 18 %, long scoreboard 16 %), not by issue
// slots.  The exact form stays.
template <int D>  // D = 1 (CLS) + number of signals
__global__ void __launch_bounds__(kMixThreads, 1) epoch_mixer_kernel(const MixerArgs p) {
  constexpr int R = 16 * D;
  extern __shared__ __align__(16) uint8_t smem[];
  float* sX = reinterpret_cast<float*>(smem);
  __half* sA = reinterpret_cast<__half*>(smem + (size_t)R * kMixLdX * 4);
  __half* sQ = sA + (size_t)R * kMixLdA;  // QKV [R][kMixLdQ] and later FFN hidden [R][kMixLdH]
  uint8_t* sMask = reinterpret_cast<uint8_t*>(sQ + (size_t)R * kMixLdH);  // [16][8]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_tiles = (p.n_epochs + kMixEp - 1) / kMixEp;

#pragma unroll 1
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int n0 = tile * kMixEp;
    __syncthreads();  // previous tile fully consumed
    // ---- masks + token load ----
    if (tid < 16 * D) {
      const int e = tid & 15, j = tid >> 4;
      const int n = n0 + e;
      uint8_t m = 0;
      if (n >= p.n_epochs) m = (j > 0);
      else if (j > 0) m = p.row_mask[j - 1] != nullptr ? p.row_mask[j - 1][n / p.S] : 0;
      sMask[e * 8 + j] = m;
    }
    __syncthreads();
    for (int idx = tid; idx < R * 16; idx += kMixThreads) {  // 16 x 8-half chunks per row
      const int row = idx >> 4, ck = idx & 15;
      const int j = row >> 4, e = row & 15;
      float v[8];
      if (j == 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = __ldg(p.cls + ck * 8 + k);
      } else if (sMask[e * 8 + j]) {
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = 0.0f;  // wav2sleep.py:320
      } else {
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(p.z[j - 1] + (size_t)(n0 + e) * kMixF) + ck);
        const uint32_t* uu = reinterpret_cast<const uint32_t*>(&u);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 f = unpack_h2(uu[q]);
          v[2 * q] = f.x;
          v[2 * q + 1] = f.y;
        }
      }
      float4* dst = reinterpret_cast<float4*>(sX + (size_t)row * kMixLdX + ck * 8);
      dst[0] = make_float4(v[0], v[1], v[2], v[3]);
      dst[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
    __syncthreads();

#pragma unroll 1
    for (int l = 0; l < p.n_layers; ++l) {
      const MixerLayerW& W = p.layer[l];
      const bool last = (l == p.n_layers - 1);
      const int mq = last ? 1 : D;  // m-tiles that need Q / out-proj / FFN

      // ---- x -> LN1 -> sA ----
      mixer_layernorm(sX, sA, R, W.ln1_w, W.ln1_b, p.ln_eps, warp, lane);
      __syncthreads();

      // ---- QKV projection ----
      {
        auto epi = [&](int row, int col, float v0, float v1) {
          const float2 bv = __ldg(reinterpret_cast<const float2*>(W.in_b + col));
          *reinterpret_cast<uint32_t*>(sQ + (size_t)row * kMixLdQ + col) = pack_h2(v0 + bv.x, v1 + bv.y);
        };
        if (!last) {
          warp_gemm<D, 8>(sA, kMixLdA, D, W.in_w, warp * (48 / kMixWarps), 48 / kMixWarps, lane, epi);  // 48 n-tiles
        } else {
          warp_gemm<D, 8>(sA, kMixLdA, D, W.in_w, 16 + warp * (32 / kMixWarps), 32 / kMixWarps, lane, epi);  // K,V: n-tiles 16..47
          warp_gemm<D, 8>(sA, kMixLdA, 1, W.in_w, warp * (16 / kMixWarps), 16 / kMixWarps, lane, epi);  // Q of the CLS tile
        }
      }
      __syncthreads();

      // ---- attention: one (epoch, head, query token) per work item ----
      {
        const int items = mq * 16 * kMixHeads;
        for (int it = tid; it < items; it += kMixThreads) {
          const int e = it & 15, h = (it >> 4) & 7, i = it >> 7;
          const __half* qp = sQ + (size_t)(i * 16 + e) * kMixLdQ + h * kMixHd;
          float q[16];
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(qp + 2 * k));
            q[2 * k] = f.x;
            q[2 * k + 1] = f.y;
          }
          float s[D];
          float mx = -INFINITY;
#pragma unroll
          for (int j = 0; j < D; ++j) {
            const __half* kp = sQ + (size_t)(j * 16 + e) * kMixLdQ + kMixF + h * kMixHd;
            float d = 0.0f;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const float2 f = __half22float2(*reinterpret_cast<const __half2*>(kp + 2 * k));
              d = fmaf(q[2 * k], f.x, d);
              d = fmaf(q[2 * k + 1], f.y, d);
            }
            s[j] = sMask[e * 8 + j] ? -INFINITY : d * 0.25f;  // 1/sqrt(head_dim)
            mx = fmaxf(mx, s[j]);
          }
          float den = 0.0f;
#pragma unroll
          for (int j = 0; j < D; ++j) {
            s[j] = __expf(s[j] - mx);  // masked -> exp(-inf) = 0; CLS key is never masked
            den += s[j];
          }
          const float inv = 1.0f / den;
          float o[16];
#pragma unroll
          for (int k = 0; k < 16; ++k) o[k] = 0.0f;
#pragma unroll
          for (int j = 0; j < D; ++j) {
            const __half* vp = sQ + (size_t)(j * 16 + e) * kMixLdQ + 2 * kMixF + h * kMixHd;
            const float pj = s[j] * inv;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const float2 f = __half22float2(*reinterpret_cast<const __half2*>(vp + 2 * k));
              o[2 * k] = fmaf(pj, f.x, o[2 * k]);
              o[2 * k + 1] = fmaf(pj, f.y, o[2 * k + 1]);
            }
          }
          __half* op = sA + (size_t)(i * 16 + e) * kMixLdA + h * kMixHd;
#pragma unroll
          for (int k = 0; k < 8; ++k) *reinterpret_cast<uint32_t*>(op + 2 * k) = pack_h2(o[2 * k], o[2 * k + 1]);
        }
      }
      __syncthreads();

      // ---- out-proj + residual ----
      {
        auto epi = [&](int row, int col, float v0, float v1) {
          const float2 bv = __ldg(reinterpret_cast<const float2*>(W.out_b + col));
          float2* x = reinterpret_cast<float2*>(sX + (size_t)row * kMixLdX + col);
          float2 xv = *x;
          xv.x += v0 + bv.x;
          xv.y += v1 + bv.y;
          *x = xv;
        };
        warp_gemm<D, 8>(sA, kMixLdA, mq, W.out_w, warp * (16 / kMixWarps), 16 / kMixWarps, lane, epi);
      }
      __syncthreads();

      // ---- x -> LN2 -> sA ----
      mixer_layernorm(sX, sA, mq * 16, W.ln2_w, W.ln2_b, p.ln_eps, warp, lane);
      __syncthreads();

      // ---- FFN up + GELU ----
      {
        auto epi = [&](int row, int col, float v0, float v1) {
          const float2 bv = __ldg(reinterpret_cast<const float2*>(W.ff1_b + col));
          *reinterpret_cast<uint32_t*>(sQ + (size_t)row * kMixLdH + col) =
              pack_h2(gelu_erf(v0 + bv.x), gelu_erf(v1 + bv.y));
        };
        warp_gemm<D, 8>(sA, kMixLdA, mq, W.ff1_w, warp * (64 / kMixWarps), 64 / kMixWarps, lane, epi);
      }
      __syncthreads();

      // ---- FFN down + residual ----
      {
        auto epi = [&](int row, int col, float v0, float v1) {
          const float2 bv = __ldg(reinterpret_cast<const float2*>(W.ff2_b + col));
          float2* x = reinterpret_cast<float2*>(sX + (size_t)row * kMixLdX + col);
          float2 xv = *x;
          xv.x += v0 + bv.x;
          xv.y += v1 + bv.y;
          *x = xv;
        };
        warp_gemm<D, 32>(sQ, kMixLdH, mq, W.ff2_w, warp * (16 / kMixWarps), 16 / kMixWarps, lane, epi);
      }
      __syncthreads();
    }

    // ---- CLS rows -> global ----
    for (int idx = tid; idx < 16 * 16; idx += kMixThreads) {
      const int e = idx >> 4, ck = idx & 15;
      if (n0 + e < p.n_epochs) {
        const float* x = sX + (size_t)e * kMixLdX + ck * 8;
        uint4 u = make_uint4(pack_h2(x[0], x[1]), pack_h2(x[2], x[3]), pack_h2(x[4], x[5]), pack_h2(x[6], x[7]));
        *(reinterpret_cast<uint4*>(p.out + (size_t)(n0 + e) * kMixF) + ck) = u;
      }
    }
  }
}

template <int D>
inline cudaError_t launch_epoch_mixer_d(const MixerArgs& a, int sm_count, cudaStream_t stream) {
  auto kern = epoch_mixer_kernel<D>;
  constexpr size_t smem = mixer_smem_bytes<D>();
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  const int n_tiles = (a.n_epochs + kMixEp - 1) / kMixEp;
  const int grid = n_tiles < sm_count ? n_tiles : sm_count;
  kern<<<grid, kMixThreads, smem, stream>>>(a);
  return cudaGetLastError();
}

inline cudaError_t launch_epoch_mixer(const MixerArgs& a, int n_sig, int sm_count, cudaStream_t stream) {
  switch (n_sig) {
    case 1: return launch_epoch_mixer_d<2>(a, sm_count, stream);
    case 2: return launch_epoch_mixer_d<3>(a, sm_count, stream);
    case 3: return launch_epoch_mixer_d<4>(a, sm_count, stream);
    case 4: return launch_epoch_mixer_d<5>(a, sm_count, stream);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace w2s
