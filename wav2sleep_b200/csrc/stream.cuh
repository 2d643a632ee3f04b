// Streaming step of a causal SequenceCNN + classifier: R new epochs of N independent streams per launch, with the
// history each dilated layer needs carried in ring buffers in HBM (w2s_gen_seq_stream_step, wav2sleep_b200/streaming.py).
//
// Reference restated: SequenceCNN.forward (models/wav2sleep.py:379-390), DilatedConvBlock (models/blocks.py:115-126),
// ConvLayer1D in causal mode (blocks.py:150-152, 173-186: output t reads inputs t - (k-1-i)*d, i < k, zero before 0),
// Wav2Sleep.classifier (models/wav2sleep.py:41, 66).  Eval semantics: running BatchNorm statistics, no dropout.
//
// Ring of layer l (dilation d, M = (k-1)*d rows of F floats per stream): the input row of epoch e sits in slot e mod M.
// Tap i < k-1 of epoch e reads epoch e - (k-1-i)*d = slot (e + i*d) mod M; tap 0 is the slot epoch e overwrites, so
// every tap is read before the new row is written.  Zero rings are the causal zero padding of the full forward.
//
// Parallelism: one CTA owns a tile of TS = G * spt streams.  Thread (g, co), g < G = 256 / F, computes output channel co
// of streams g, g + G, ... (spt accumulators).  Tap rows of the tile, the block input and the layer output live in shared
// memory; each layer's weights stream through shared memory in chunks of `cc` input channels and serve every stream of
// the tile.  fp32 throughout, no tensor cores (M is the stream count).  A stream's arithmetic does not depend on the
// tile it sits in, on R or on the other streams.
#pragma once
#include "general.cuh"

namespace w2s {
namespace gen {

constexpr int kStreamThreads = 256;
constexpr int kStreamMaxAcc = 8;  // streams per thread
constexpr int kStageLoads = 8;    // global loads in flight per thread while staging weights / ring taps

// dst(i, src(i)) for i < n over the CTA: each thread issues kStageLoads independent loads before their shared stores, so
// a chunk costs about one L2 round trip instead of one per element a thread copies.
template <class Src, class Dst>
W2S_DEVINL void staged_copy(int n, Src src, Dst dst) {
  for (int i0 = threadIdx.x; i0 < n; i0 += kStageLoads * blockDim.x) {
    float v[kStageLoads];
#pragma unroll
    for (int u = 0; u < kStageLoads; ++u) {
      const int i = i0 + u * blockDim.x;
      if (i < n) v[u] = src(i);
    }
#pragma unroll
    for (int u = 0; u < kStageLoads; ++u) {
      const int i = i0 + u * blockDim.x;
      if (i < n) dst(i, v[u]);
    }
  }
}

struct SeqStreamArgs {
  w2s_gen_seq_stream_desc d;
  const float* x; float* logits;
  int N, R; long long pos;
  int G, spt, cc;  // thread groups, streams per thread, input channels per weight chunk
};

// shared floats of one CTA: taps [TS][k][F], y [TS][F], block input [TS][F], weight chunk [cc * k][F | 1]
inline size_t seq_stream_smem_floats(int F, int k, int TS, int cc) {
  return (size_t)TS * (k + 2) * F + (size_t)cc * k * (F | 1);
}

__global__ void __launch_bounds__(kStreamThreads) seq_stream_kernel(const SeqStreamArgs p) {
  extern __shared__ float sm[];
  const w2s_gen_seq_stream_desc& d = p.d;
  const int F = d.feature_dim, k = d.kernel_size, G = p.G, spt = p.spt, TS = G * spt, ld = F | 1;
  float* taps = sm;
  float* y = taps + (size_t)TS * k * F;
  float* bin = y + (size_t)TS * F;
  float* ws = bin + (size_t)TS * F;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;
  const int g = tid / F, co = tid % F;
  const bool active = g < G;
  const long long s0 = (long long)blockIdx.x * TS;
  const int nvalid = (int)min((long long)TS, (long long)p.N - s0);
  const int n_layers = d.n_blocks * d.n_dilations;
  const long long rows = (long long)d.n_blocks * (k - 1) * ((1LL << d.n_dilations) - 1);  // ring rows per stream

  for (size_t i = tid; i < (size_t)TS * (k + 2) * F; i += blockDim.x) sm[i] = 0.0f;  // tail streams stay zero

  for (int r = 0; r < p.R; ++r) {
    const long long e = p.pos + r;
    __syncthreads();  // the previous epoch's classifier has read its rows
    for (int i = tid; i < nvalid * F; i += blockDim.x) {
      const int s = i / F, f = i % F;
      const float v = p.x[((size_t)(s0 + s) * p.R + r) * F + f];
      taps[((size_t)s * k + k - 1) * F + f] = v;
      bin[(size_t)s * F + f] = v;
    }
    long long ring_off = 0;
    for (int l = 0; l < n_layers; ++l) {
      const w2s_gen_seq_stream_layer& L = d.layer[l];
      const int j = l % d.n_dilations, dil = 1 << j, M = (k - 1) * dil;
      __syncthreads();  // the layer input is in taps[s][k-1]
      if (M > 0) {
        float* ring = d.ring + ring_off * F;
        const int km1 = k - 1;
        staged_copy(
            nvalid * km1 * F,
            [=](int i) {
              const int f = i % F, t = (i / F) % km1, s = i / (F * km1);
              return ring[((size_t)(s0 + s) * rows + (e + (long long)t * dil) % M) * F + f];
            },
            [=](int i, float v) {
              const int f = i % F, t = (i / F) % km1, s = i / (F * km1);
              taps[((size_t)s * k + t) * F + f] = v;
            });
        __syncthreads();  // every tap is read before the oldest slot is overwritten
        const long long slot = e % M;
        for (int i = tid; i < nvalid * F; i += blockDim.x) {
          const int s = i / F, f = i % F;
          ring[((size_t)(s0 + s) * rows + slot) * F + f] = taps[((size_t)s * k + k - 1) * F + f];
        }
      }
      ring_off += M;

      // conv: acc[i] = bias[co] + sum_{ci, t} taps[s_i][t][ci] * w[co, ci, t]
      float acc[kStreamMaxAcc];
      const float b0 = (active && L.bias) ? L.bias[co] : 0.0f;
#pragma unroll
      for (int i = 0; i < kStreamMaxAcc; ++i) acc[i] = b0;
      for (int c0 = 0; c0 < F; c0 += p.cc) {
        const int nc = min(p.cc, F - c0), kc = nc * k;
        __syncthreads();  // the previous chunk is consumed
        const float* wl = L.w;
        staged_copy(
            F * kc, [=](int i) { return wl[((size_t)(i / kc) * F + c0) * k + i % kc]; },
            [=](int i, float v) { ws[(size_t)(i % kc) * ld + i / kc] = v; });
        __syncthreads();
        if (active) {
          for (int cc = 0; cc < nc; ++cc) {
            for (int t = 0; t < k; ++t) {
              const float w = ws[(size_t)(cc * k + t) * ld + co];
              const float* a = taps + (size_t)t * F + c0 + cc;
#pragma unroll
              for (int i = 0; i < kStreamMaxAcc; ++i)
                if (i < spt) acc[i] = fmaf(a[(size_t)(g + i * G) * k * F], w, acc[i]);
            }
          }
        }
      }
      if (active) {
#pragma unroll
        for (int i = 0; i < kStreamMaxAcc; ++i)
          if (i < spt) y[(size_t)(g + i * G) * F + co] = acc[i];
      }
      __syncthreads();

      // norm -> activation (-> + block input -> activation at the block end); one warp per stream row
      const bool block_end = j == d.n_dilations - 1;
      for (int s = warp; s < TS; s += nwarps) {
        float* row = y + (size_t)s * F;
        float mean = 0.0f, rstd = 1.0f;
        if (d.norm == W2S_SEQ_NORM_LAYER || d.norm == W2S_SEQ_NORM_RMS) {  // as rownorm_kernel
          if (d.norm == W2S_SEQ_NORM_LAYER) {
            float sum = 0.0f;
            for (int c = lane; c < F; c += 32) sum += row[c];
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            mean = sum / (float)F;
          }
          float q = 0.0f;
          for (int c = lane; c < F; c += 32) {
            const float dv = row[c] - mean;
            q = fmaf(dv, dv, q);
          }
          for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
          rstd = 1.0f / sqrtf(q / (float)F + d.eps);
        }
        for (int c = lane; c < F; c += 32) {
          float v = row[c];
          if (d.norm == W2S_SEQ_NORM_BATCH) {  // eval BatchNorm1d, constants as norm_consts_kernel
            const double rs = 1.0 / sqrt((double)L.running_var[c] + (double)d.eps);
            const double w = L.norm_w ? (double)L.norm_w[c] : 1.0, b = L.norm_b ? (double)L.norm_b[c] : 0.0;
            v *= (float)(rs * w);
            v += (float)(b - (double)L.running_mean[c] * rs * w);
          } else if (d.norm != W2S_SEQ_NORM_NONE) {
            v = (v - mean) * rstd * (L.norm_w ? L.norm_w[c] : 1.0f) + (L.norm_b ? L.norm_b[c] : 0.0f);
          }
          v = activate(v, d.act);
          if (block_end) {
            v = activate(v + bin[(size_t)s * F + c], d.act);
            bin[(size_t)s * F + c] = v;
          }
          taps[((size_t)s * k + k - 1) * F + c] = v;
        }
      }
    }
    __syncthreads();

    // classifier, as the 1-tap conv of the general path: logits = b + sum_f h[f] * W[c, f]
    const int C = d.n_classes;
    for (int i = tid; i < nvalid * C; i += blockDim.x) {
      const int s = i / C, c = i % C;
      const float* h = taps + ((size_t)s * k + k - 1) * F;
      const float* w = d.head_w + (size_t)c * F;
      float acc = d.head_b ? d.head_b[c] : 0.0f;
      for (int f = 0; f < F; ++f) acc = fmaf(h[f], w[f], acc);
      p.logits[((size_t)(s0 + s) * p.R + r) * C + c] = acc;
    }
  }
}

}  // namespace gen
}  // namespace w2s
