// Implicit-GEMM 1-D convolution on tcgen05 tensor cores (sm_100a), channels-last fp16 activations.
//
// One kernel template covers every dense contraction of the wav2sleep forward:
//   * encoder ConvLayer1D  k=3, stride 1|2            (reference models/blocks.py:173-186, 25-44)
//   * encoder 1x1 stride-2 residual "downsample"      (blocks.py:46-53) as a 2nd accumulator of conv1
//   * encoder time-distributed Linear(4C -> F) + GELU (models/wav2sleep.py:261-265) as taps=4, stride=4
//   * sequence-mixer dilated conv k=7 + ConvLayerNorm + GELU (+ residual + GELU [+ classifier])
//                                                     (blocks.py:93-126, utils.py:9-23, wav2sleep.py:66)
//
// GEMM view: M = output positions (128 per UMMA), N = COUT, K = TAPS * CIN.
// A (activations) is staged by the CTA's threads - not TMA - because the whole-night InstanceNorm of the
// producing layer (utils.py:89-92, eps 1e-2) can only be applied by the consumer: the prologue turns the stored
// pre-norm fp16 values into GELU((y - mu) * rstd) [optionally GELU(. + residual)] on the way to shared memory.
// Staging layout is [stride phase][16-byte channel chunk][row][8 halfs] ("chunk-major", no swizzle), so a conv
// tap is just a row offset of the UMMA shared-memory descriptor: im2col costs nothing.
// B (weights) is pre-packed on the host as [tap][chunk][cout][8 halfs] and copied linearly.
// Accumulators live in TMEM; the epilogue reads them with tcgen05.ld (thread == output position) and
//   EPI_STATS     : stores pre-norm fp16 + accumulates sum / sum-of-squares per (sample, channel)
//   EPI_BIAS_GELU : + bias, exact GELU, stores fp16
//   EPI_LN_GELU   : LayerNorm over the 128 channels of the thread's row, affine, GELU
//   EPI_LN_GELU_RES: ... + block input, GELU, optional fused classifier head
//   EPI_ACT_BWD   : training data-gradient conv fused with the backward through the producing layer's activation:
//                   da = acc (+ res); x_hat = IN(ab_y); [block outputs: s = GELU(x_hat) + ab_r, ds = da GELU'(s), dr = ds]
//                   d(x_hat) = ds GELU'(x_hat) -> out; the activated tensor itself -> ab_a (operand of the weight
//                   gradient); sum d(x_hat), sum d(x_hat) x_hat per (sample, channel) -> out_stats (fp64)
//   EPI_PLAIN     : (+ bias) (+ residual tensor) -> fp16, output rows at o*out_stride + out_offset (plain GEMMs and
//                   data-gradient convolutions of the training path)
// Training prologue PRO_DNORM (data-gradient convs): the conv input is the gradient dy of the layer's pre-norm output,
//   which is the InstanceNorm backward of d(x_hat): dy = rstd (d(x_hat) - mean(d x_hat) - x_hat mean(d x_hat . x_hat)),
//   x_hat = (y - mu) rstd.  It is computed on the way to shared memory from `in` = d(x_hat) and `in_res` = y (the layer's
//   stored forward output) with the per-(sample, channel) constants from in_stats (sum y, sum y^2) and dn_sums
//   (sum d x_hat, sum d x_hat . x_hat); each tile also writes the dy rows it owns to dn_out, for the weight-gradient
//   GEMM that follows.  dn_upsample: the layer was a stride-2 conv - its gradient enters the (stride-1) data-gradient
//   conv zero-stuffed: input row i = source row i / 2 for even i, zero for odd i.
#pragma once
#include <cstring>
#include "common.cuh"

namespace w2s {

enum : int { PRO_NONE = 0, PRO_NORM = 1, PRO_NORM_RES = 2, PRO_FIR = 3, PRO_NORM_RES_X = 4, PRO_DNORM = 5 };
enum : int { EPI_STATS = 0, EPI_BIAS_GELU = 1, EPI_LN_GELU = 2, EPI_LN_GELU_RES = 3, EPI_PLAIN = 4, EPI_ACT_BWD = 5 };

struct ConvArgs {
  // input side
  const act_t* in;        // [B, L_in, CIN]  pre-norm (PRO_NORM*) or final (PRO_NONE)
  const act_t* in_res;    // [B, L_in, CIN]  residual branch of the producing block (PRO_NORM_RES)
  const double* in_stats; // [B, CIN, 2]     sum, sum of squares over L_in of `in` (fp64: order-independent)
  const act_t* w;         // packed [TAPS][CIN/8][COUT][8]  (SPLIT: hi block followed by lo block)
  const act_t* w_ds;      // packed [CIN/8][COUT][8] (HAS_DS; SPLIT: hi then lo)
  // output side
  act_t* out;             // [B, L_out, COUT]
  act_t* out_ds;          // [B, L_out/2, COUT] (HAS_DS)
  double* out_stats;      // [B, COUT, 2] (EPI_STATS), must be zeroed by the caller
  const uint8_t* row_mask;  // [B] non-zero => sample has no such signal: skip (may be null)
  const float* bias;      // [COUT] (EPI_BIAS_GELU)
  const float* ln_w;      // [COUT] (EPI_LN_*)
  const float* ln_b;      // [COUT]
  const act_t* res;       // [B, L_out, COUT] block input (EPI_LN_GELU_RES)
  const float* head_w;    // [n_classes, COUT] or null
  const float* head_b;    // [n_classes]
  float* logits;          // [B, L_out, n_classes]
  int n_classes;
  int L_in, L_out;
  int stride_log2;        // stride = 1 << stride_log2
  int dil, pad;
  float in_eps;           // InstanceNorm eps (1e-2)
  float ln_eps;           // ConvLayerNorm eps (1e-5)
  int out_stride;         // EPI_PLAIN: output row = o * out_stride + out_offset inside a sample of out_rows rows
  int out_offset;
  int out_rows;
  // EPI_ACT_BWD: the producing layer's pre-norm output / residual branch / statistics, and the extra outputs
  const act_t* ab_y;      // [B, L_out, COUT]
  const act_t* ab_r;      // [B, L_out, COUT] or null (plain layer)
  const double* ab_stats; // [B, COUT, 2] sum, sumsq of ab_y over L_out
  act_t* ab_a;            // [B, L_out, COUT] activated tensor (may be null)
  act_t* ab_dr;           // [B, L_out, COUT] gradient of the residual branch (ab_r != null)
  float ab_eps;
  // streaming kernel, block-0 fusion (PRO_FIR / PRO_NORM_RES_X): the raw signal and the Cin = 1 weights of block 0
  const float* x_raw;     // [B, T_raw] fp32
  const float* w_first;   // [16, 3]
  const float* w_first_ds;  // [16]
  int T_raw;
  // PRO_DNORM
  const double* dn_sums;  // [B, CIN, 2] sum d(x_hat), sum d(x_hat) x_hat over the layer's output length
  act_t* dn_out;          // [B, L_in, CIN] dy (zero-stuffed when dn_upsample)
  int dn_upsample;
  // Profiling experiments only (W2S_DEBUG_FLAGS in the environment; 0 in production, results are wrong otherwise):
  //   1 skip the lo-operand MMAs, 2 skip all MMAs, 4 skip GELU, 8 skip epilogue stores, 16 skip epilogue TMEM loads,
  //   32 skip the transform, 64 record timestamps / per-role wait cycles (results stay correct), 128 / 256 skip only the
  //   A_lo / W_lo MMA, 512 / 1024 the same for CIN = 32 layers only.
  int debug_flags;
};

// Paired launch: two encoders with identical layer shapes (ECG + PPG, ABD + THX) run a layer in ONE launch - the first
// half of the grid works on group 0, the second half on group 1.  Only the tensors differ between the groups: the second
// group's pointers ride in this block (ngroups == 1: ignored), every scalar of ConvArgs is shared.  Halves the number of
// stream-kernel launches of a forward and with it the per-launch fixed cost (set-up, pipeline fill, drain, exit spread:
// ~8 us of every CTA's life, profiles/r02_fixed_cost_small_layers.txt), and gives each CTA twice the tiles per launch.
struct ConvGroup2 {
  const act_t* in;
  const act_t* in_res;
  const double* in_stats;
  const act_t* w;
  const act_t* w_ds;
  act_t* out;
  act_t* out_ds;
  double* out_stats;
  const uint8_t* row_mask;
  const float* x_raw;
  const float* w_first;
  const float* w_first_ds;
  int ngroups;
};
// Kernels that are already at their register cap stay single-group (the second group's pointers would be selected into
// registers: 72 -> 330 bytes of spills in the staged two-accumulator epilogue of the 128-channel conv1 kernels).
__host__ __device__ constexpr bool stream_pairable(int cout, bool has_ds) { return !(cout == 128 && has_ds); }
inline ConvGroup2 conv_group2(const ConvArgs* a) {
  ConvGroup2 g;
  memset(&g, 0, sizeof(g));
  g.ngroups = 1;
  if (a != nullptr) {
    g.in = a->in; g.in_res = a->in_res; g.in_stats = a->in_stats; g.w = a->w; g.w_ds = a->w_ds;
    g.out = a->out; g.out_ds = a->out_ds; g.out_stats = a->out_stats; g.row_mask = a->row_mask;
    g.x_raw = a->x_raw; g.w_first = a->w_first; g.w_first_ds = a->w_first_ds;
    g.ngroups = 2;
  }
  return g;
}

constexpr int kConvThreads = 256;

template <int COUT>
struct ConvTile {
  static constexpr int MT = 128 / COUT;    // 128-row UMMA sub-tiles per CTA
  static constexpr int POS = 128 * MT;     // output positions per CTA
};

// Rows of staged input per stride phase for a CTA tile.
__host__ __device__ inline int conv_rows_per_phase(int pos, int stride, int taps, int dil) {
  const int R = (pos - 1) * stride + (taps - 1) * dil + 1;
  return (R + stride - 1) / stride;
}
// SPLIT: operands are carried as fp16 hi + fp16 lo (A = A_hi + A_lo, W = W_hi + W_lo) and the product is
// A_hi*W_hi + A_lo*W_hi + A_hi*W_lo: ~22-bit operands on the fp16 tensor pipe.  Default rule: the 16-channel layers,
// whose operand rounding dominates the logit error (tools/emulate_16bit.py: cardio mean error 1.9e-3 without any split,
// 1.5e-3 with the 16-channel layers split, 1.3e-3 with the 32-channel layers split as well - not worth 3x the MMAs
// on 27 % of the step).  Deep encoders (wide storage) override it per layer up to 64 channels.
template <int CIN, int COUT>
struct ConvSplit {
  static constexpr bool value = (CIN <= 16 && COUT <= 16);
};
constexpr int kConvCtlBytes = 16 + 2 * 128 * 4 + 2 * 512 * 4 + 4 * 128 * 4;  // barrier+tmem slot, scale/shift, stats partials, PRO_DNORM constants
template <int CIN, int COUT, int GT, bool HAS_DS, bool SPLIT>
__host__ __device__ inline size_t conv_smem_bytes(int stride, int taps, int dil) {
  const int rp = conv_rows_per_phase(ConvTile<COUT>::POS, stride, taps, dil);
  size_t a = (size_t)stride * (CIN / 8) * rp * 16;
  size_t b = (size_t)(GT + (HAS_DS ? 1 : 0)) * (CIN / 8) * COUT * 16;
  return (SPLIT ? 2 : 1) * (a + b) + kConvCtlBytes;
}

// BF16OP (measurement hook, w2s_set_conv_impl(3)): the MMA operands are bf16 instead of fp16 - activated inputs are
// rounded to bf16 in the prologue, the weights come packed as bf16, the instruction descriptor selects bf16 A / B.
// Storage stays fp16.  Evidence for the fp16-over-bf16 decision on the hardware itself (tests/test_kernels_gpu.py).
template <int CIN, int COUT, int TAPS, int GT /*taps resident per weight group*/, int PRO, int EPI, bool HAS_DS,
          bool SPLIT, bool BF16OP = false>
W2S_DEVINL void conv_igemm_body(const ConvArgs& p, const int b) {
  static_assert(!BF16OP || (!SPLIT && PRO != PRO_NONE), "bf16 operands: computed prologue, single operand");
  static_assert(!SPLIT || (GT == TAPS && PRO != PRO_NONE), "split operands: single weight group, computed prologue");
  static_assert(CIN % 16 == 0 && COUT % 16 == 0 && COUT <= 128, "UMMA shape");
  static_assert(EPI == EPI_STATS || EPI == EPI_PLAIN || EPI == EPI_ACT_BWD || COUT == 128,
                "row-wise epilogues need the full channel dim in one tile");
  constexpr int CH = CIN / 8;                 // 16-byte chunks per input row
  constexpr int MT = ConvTile<COUT>::MT;
  constexpr int POS = ConvTile<COUT>::POS;
  constexpr int KSTEPS = CIN / 16;            // UMMA K=16 steps per tap
  constexpr int NGROUPS = (TAPS + GT - 1) / GT;
  constexpr uint32_t TMEM_COLS = HAS_DS ? 256 : 128;
  constexpr uint32_t IDESC = umma_idesc_f16(128, COUT, BF16OP);

  if (p.row_mask != nullptr && p.row_mask[b]) return;
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int stride = 1 << p.stride_log2;
  const int o0 = blockIdx.x * POS;            // first output position of this tile
  const int i0 = o0 * stride - p.pad;         // input row staged at u = 0
  const int R = (POS - 1) * stride + (TAPS - 1) * p.dil + 1;
  const int Rp = (R + stride - 1) >> p.stride_log2;

  extern __shared__ __align__(128) uint8_t smem[];
  const size_t a_bytes = (size_t)stride * CH * Rp * 16;
  constexpr size_t b_bytes = (size_t)(GT + (HAS_DS ? 1 : 0)) * CH * COUT * 16;
  uint8_t* sA = smem;                                  // hi (or only) activations
  uint8_t* sAlo = sA + a_bytes;                        // lo activations (SPLIT)
  uint8_t* sB = sA + (SPLIT ? 2 : 1) * a_bytes;        // hi weights [GT taps (+ds)][CH][COUT][8]
  uint8_t* sBlo = sB + b_bytes;                        // lo weights (SPLIT)
  uint8_t* sCtl = sB + (SPLIT ? 2 : 1) * b_bytes;
  uint64_t* bar = reinterpret_cast<uint64_t*>(sCtl);            // 8 B
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sCtl + 8);  // 4 B
  float* sScale = reinterpret_cast<float*>(sCtl + 16);          // [128]
  float* sShift = sScale + 128;                                 // [128]
  float* sPartSum = sShift + 128;                               // [8 warps][4 units][16 ch]
  float* sPartSq = sPartSum + 512;
  float* sDn = sPartSq + 512;                                   // PRO_DNORM: [mean | rstd | m1 | m2][128]
  (void)sDn;

  // ---------------- setup ----------------
  if (warp == 0) tmem_alloc(tmem_slot, TMEM_COLS);
  if (tid == 32) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  if (PRO == PRO_DNORM && tid >= 64 && tid < 64 + CIN) {
    const int c = tid - 64;
    const int Ls = p.dn_upsample ? (p.L_in >> 1) : p.L_in;  // length of the layer output the statistics run over
    float mean, rstd;
    in_consts(p.in_stats, b, CIN, c, Ls, p.in_eps, mean, rstd);
    const float invL = 1.0f / (float)Ls;
    sDn[c] = mean;
    sDn[128 + c] = rstd;
    sDn[256 + c] = (float)p.dn_sums[((size_t)b * CIN + c) * 2] * invL;
    sDn[384 + c] = (float)p.dn_sums[((size_t)b * CIN + c) * 2 + 1] * invL;
  }
  if (PRO != PRO_NONE && PRO != PRO_DNORM && tid >= 64 && tid < 64 + CIN) {
    const int c = tid - 64;
    const double s0 = p.in_stats[((size_t)b * CIN + c) * 2 + 0];
    const double s1 = p.in_stats[((size_t)b * CIN + c) * 2 + 1];
    const double inv_len = 1.0 / (double)p.L_in;
    const double mean = s0 * inv_len;
    const double var = fmax(s1 * inv_len - mean * mean, 0.0);  // biased variance (InstanceNorm1d)
    const float rstd = (float)(1.0 / sqrt(var + (double)p.in_eps));
    sScale[c] = rstd;
    sShift[c] = (float)(-mean) * rstd;
  }
  if (EPI == EPI_ACT_BWD && tid >= 64 && tid < 64 + COUT) {  // InstanceNorm constants of the layer that produced ab_y
    float mean, rstd;
    in_consts(p.ab_stats, b, COUT, tid - 64, p.L_out, p.ab_eps, mean, rstd);
    sScale[tid - 64] = rstd;
    sShift[tid - 64] = mean;
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  // ---------------- prologue: global -> (norm, GELU) -> smem A ----------------
  if constexpr (PRO == PRO_DNORM) {
    // InstanceNorm backward on the way in (see the header): 4 row chunks in flight per thread, two tensors each
    const int cch = tid & (CH - 1);
    float mean[8], rstd[8], m1[8], m2[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      mean[k] = sDn[cch * 8 + k];
      rstd[k] = sDn[128 + cch * 8 + k];
      m1[k] = sDn[256 + cch * 8 + k];
      m2[k] = sDn[384 + cch * 8 + k];
    }
    const int total = R * CH;
    const int up = p.dn_upsample;
    const int Ls = up ? (p.L_in >> 1) : p.L_in;
    const act_t* gb = p.in + (size_t)b * Ls * CIN;        // d(x_hat)
    const act_t* yb = p.in_res + (size_t)b * Ls * CIN;    // y
    act_t* dyb = p.dn_out + (size_t)b * p.L_in * CIN;
    constexpr int UN = 4;
    for (int base = tid; base < total; base += kConvThreads * UN) {
      uint4 g[UN], y[UN];
#pragma unroll
      for (int k = 0; k < UN; ++k) {
        const int id = base + k * kConvThreads;
        const int i = i0 + id / CH;
        g[k] = y[k] = make_uint4(0u, 0u, 0u, 0u);
        if (id < total && i >= 0 && i < p.L_in && !(up && (i & 1))) {
          const size_t off = (size_t)(up ? (i >> 1) : i) * CIN + cch * 8;
          g[k] = __ldg(reinterpret_cast<const uint4*>(gb + off));
          y[k] = __ldg(reinterpret_cast<const uint4*>(yb + off));
        }
      }
#pragma unroll
      for (int k = 0; k < UN; ++k) {
        const int id = base + k * kConvThreads;
        if (id >= total) break;
        const int u = id / CH;
        const int i = i0 + u;
        uint4 o = make_uint4(0u, 0u, 0u, 0u);
        if (i >= 0 && i < p.L_in && !(up && (i & 1))) {
          const uint32_t* gg = reinterpret_cast<const uint32_t*>(&g[k]);
          const uint32_t* yy = reinterpret_cast<const uint32_t*>(&y[k]);
          uint32_t* oo = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float2 gv = unpack_h2(gg[q]), yv = unpack_h2(yy[q]);
            const float xh0 = (yv.x - mean[2 * q]) * rstd[2 * q], xh1 = (yv.y - mean[2 * q + 1]) * rstd[2 * q + 1];
            oo[q] = pack_h2(rstd[2 * q] * (gv.x - m1[2 * q] - xh0 * m2[2 * q]),
                            rstd[2 * q + 1] * (gv.y - m1[2 * q + 1] - xh1 * m2[2 * q + 1]));
          }
        }
        const int phase = u & (stride - 1);
        const int row = u >> p.stride_log2;
        *reinterpret_cast<uint4*>(sA + ((size_t)(phase * CH + cch) * Rp + row) * 16) = o;
        // rows this tile owns (the POS input rows aligned with its outputs; halo rows belong to the neighbours)
        if (u >= p.pad && u < p.pad + POS && i < p.L_in) *reinterpret_cast<uint4*>(dyb + (size_t)i * CIN + cch * 8) = o;
      }
    }
  } else {
    const int cch = tid & (CH - 1);  // this thread's channel chunk is fixed (256 % CH == 0)
    float sc[8], sh[8];
    if (PRO != PRO_NONE) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        sc[k] = sScale[cch * 8 + k];
        sh[k] = sShift[cch * 8 + k];
      }
    }
    const int total = R * CH;
    const act_t* inb = p.in + (size_t)b * p.L_in * CIN;
    const act_t* resb = (PRO == PRO_NORM_RES) ? p.in_res + (size_t)b * p.L_in * CIN : nullptr;
    constexpr int UN = (PRO == PRO_NORM_RES) ? 4 : 8;
    for (int base = tid; base < total; base += kConvThreads * UN) {
      uint4 y[UN], r[UN];
#pragma unroll
      for (int k = 0; k < UN; ++k) {
        const int id = base + k * kConvThreads;
        const int u = id / CH;
        const int i = i0 + u;
        y[k] = make_uint4(0u, 0u, 0u, 0u);
        if (PRO == PRO_NORM_RES) r[k] = make_uint4(0u, 0u, 0u, 0u);
        if (id < total && i >= 0 && i < p.L_in) {
          const size_t off = (size_t)i * CIN + cch * 8;
          y[k] = __ldg(reinterpret_cast<const uint4*>(inb + off));
          if (PRO == PRO_NORM_RES) r[k] = __ldg(reinterpret_cast<const uint4*>(resb + off));
        }
      }
#pragma unroll
      for (int k = 0; k < UN; ++k) {
        const int id = base + k * kConvThreads;
        if (id >= total) break;
        const int u = id / CH;
        const int i = i0 + u;
        uint4 o = y[k];
        uint4 olo = make_uint4(0u, 0u, 0u, 0u);
        if (PRO != PRO_NONE) {
          if (i >= 0 && i < p.L_in) {  // zero padding applies to the *activated* signal
            uint32_t* yy = reinterpret_cast<uint32_t*>(&y[k]);
            uint32_t* rr = reinterpret_cast<uint32_t*>(&r[k]);
            uint32_t* oo = reinterpret_cast<uint32_t*>(&o);
            uint32_t* ol = reinterpret_cast<uint32_t*>(&olo);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              float2 v = unpack_h2(yy[q]);
              float a0 = gelu_fast(fmaf(v.x, sc[2 * q], sh[2 * q]));
              float a1 = gelu_fast(fmaf(v.y, sc[2 * q + 1], sh[2 * q + 1]));
              if (PRO == PRO_NORM_RES) {
                float2 rv = unpack_h2(rr[q]);
                a0 = gelu_fast(a0 + rv.x);
                a1 = gelu_fast(a1 + rv.y);
              }
              oo[q] = BF16OP ? pack_bf2(a0, a1) : pack_h2(a0, a1);
              if (SPLIT) {
                const float2 hi = unpack_h2(oo[q]);
                ol[q] = pack_h2(a0 - hi.x, a1 - hi.y);
              }
            }
          }
        }
        const int phase = u & (stride - 1);
        const int row = u >> p.stride_log2;
        const size_t soff = ((size_t)(phase * CH + cch) * Rp + row) * 16;
        *reinterpret_cast<uint4*>(sA + soff) = o;
        if (SPLIT) *reinterpret_cast<uint4*>(sAlo + soff) = olo;
      }
    }
  }

  // ---------------- main loop over weight groups ----------------
  uint32_t parity = 0;
#pragma unroll 1
  for (int g = 0; g < NGROUPS; ++g) {
    const int t_begin = g * GT;
    const int t_end = (t_begin + GT < TAPS) ? t_begin + GT : TAPS;
    {  // weights of this tap group -> smem B (linear copy of the packed layout)
      const int n16 = (t_end - t_begin) * CH * COUT;
      const uint4* src = reinterpret_cast<const uint4*>(p.w) + (size_t)t_begin * CH * COUT;
      uint4* dst = reinterpret_cast<uint4*>(sB);
      for (int k = tid; k < n16; k += kConvThreads) dst[k] = __ldg(src + k);
      if (SPLIT) {
        uint4* dlo = reinterpret_cast<uint4*>(sBlo);
        for (int k = tid; k < n16; k += kConvThreads) dlo[k] = __ldg(src + (size_t)TAPS * CH * COUT + k);
      }
      if (HAS_DS && g == 0) {
        const uint4* srcd = reinterpret_cast<const uint4*>(p.w_ds);
        uint4* dstd = dst + (size_t)GT * CH * COUT;
        for (int k = tid; k < CH * COUT; k += kConvThreads) dstd[k] = __ldg(srcd + k);
        if (SPLIT) {
          uint4* dlo = reinterpret_cast<uint4*>(sBlo) + (size_t)GT * CH * COUT;
          for (int k = tid; k < CH * COUT; k += kConvThreads) dlo[k] = __ldg(srcd + (size_t)CH * COUT + k);
        }
      }
    }
    fence_proxy_async_smem();
    __syncthreads();

    if (tid == 0) {
      tc_fence_after_sync();
      const uint32_t a_base = smem_u32(sA);
      const uint32_t b_base = smem_u32(sB);
      const uint32_t a_lo_base = smem_u32(sAlo);
      const uint32_t b_lo_base = smem_u32(sBlo);
      (void)a_lo_base;
      (void)b_lo_base;
      const uint32_t lbo_a = (uint32_t)Rp * 16;
      constexpr uint32_t lbo_b = COUT * 16;
#pragma unroll 1
      for (int j = 0; j < MT; ++j) {
        for (int t = t_begin; t < t_end; ++t) {
          const int uoff = t * p.dil;
          const int phase = uoff & (stride - 1);
          const int rowoff = (uoff >> p.stride_log2) + j * 128;
#pragma unroll
          for (int kk = 0; kk < KSTEPS; ++kk) {
            const uint32_t a_off = ((uint32_t)(phase * CH + 2 * kk) * Rp + rowoff) * 16;
            const uint32_t b_off = (uint32_t)((t - t_begin) * CH + 2 * kk) * COUT * 16;
            const uint64_t da = umma_smem_desc(a_base + a_off, lbo_a, 128);
            const uint64_t db = umma_smem_desc(b_base + b_off, lbo_b, 128);
            umma_f16(tmem_base + j * COUT, da, db, IDESC, (t > 0 || kk > 0) ? 1u : 0u);
            if (SPLIT) {
              umma_f16(tmem_base + j * COUT, umma_smem_desc(a_lo_base + a_off, lbo_a, 128), db, IDESC, 1u);
              umma_f16(tmem_base + j * COUT, da, umma_smem_desc(b_lo_base + b_off, lbo_b, 128), IDESC, 1u);
            }
          }
        }
        if (HAS_DS && g == 0) {
          // 1x1 stride-2 residual conv: centre tap rows (input position == output position of conv1);
          // computed for every row, only even positions are kept by the epilogue.
          const int rowoff = p.pad + j * 128;
#pragma unroll
          for (int kk = 0; kk < KSTEPS; ++kk) {
            const uint32_t a_off = ((uint32_t)(2 * kk) * Rp + rowoff) * 16;
            const uint32_t b_off = (uint32_t)(GT * CH + 2 * kk) * COUT * 16;
            const uint64_t da = umma_smem_desc(a_base + a_off, lbo_a, 128);
            const uint64_t db = umma_smem_desc(b_base + b_off, lbo_b, 128);
            umma_f16(tmem_base + 128 + j * COUT, da, db, IDESC, kk > 0 ? 1u : 0u);
            if (SPLIT) {
              umma_f16(tmem_base + 128 + j * COUT, umma_smem_desc(a_lo_base + a_off, lbo_a, 128), db, IDESC, 1u);
              umma_f16(tmem_base + 128 + j * COUT, da, umma_smem_desc(b_lo_base + b_off, lbo_b, 128), IDESC, 1u);
            }
          }
        }
      }
      umma_commit(bar);
    }
    mbar_wait(bar, parity);
    parity ^= 1;
    tc_fence_after_sync();
  }

  // ---------------- epilogue ----------------
  const int quad = warp & 3;   // TMEM lane quadrant this warp may read
  const int wg = warp >> 2;    // warpgroup 0/1
  const uint32_t t_lane = (uint32_t)(quad * 32) << 16;

  if (EPI == EPI_STATS) {
    act_t* outb = p.out + (size_t)b * p.L_out * COUT;
    constexpr int UNITS = MT * (COUT / 16);  // == 8
#pragma unroll 1
    for (int unit = wg; unit < UNITS; unit += 2) {
      const int j = unit / (COUT / 16);
      const int cg = unit % (COUT / 16);
      float v[16];
      tmem_ld16(tmem_base + t_lane + j * COUT + cg * 16, v);
      const int o = o0 + j * 128 + quad * 32 + lane;
      const bool valid = o < p.L_out;
      if (valid) {
        store_h16(outb + (size_t)o * COUT + cg * 16, v);
      }
      float sq[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        v[k] = valid ? v[k] : 0.0f;
        sq[k] = v[k] * v[k];
      }
      butterfly16(v, lane);
      butterfly16(sq, lane);
      if ((lane & 1) == 0) {  // one slot per (warp, unit, channel): no atomics, fixed summation order below
        const int slot = (warp * 4 + (unit >> 1)) * 16 + butterfly16_channel(lane);
        sPartSum[slot] = v[0];
        sPartSq[slot] = sq[0];
      }
    }
    if (HAS_DS) {
      act_t* dsb = p.out_ds + (size_t)b * (p.L_out >> 1) * COUT;
#pragma unroll 1
      for (int unit = wg; unit < UNITS; unit += 2) {
        const int j = unit / (COUT / 16);
        const int cg = unit % (COUT / 16);
        float v[16];
        tmem_ld16(tmem_base + t_lane + 128 + j * COUT + cg * 16, v);
        const int o = o0 + j * 128 + quad * 32 + lane;
        if (o < (p.L_out & ~1) && (o & 1) == 0) {  // out_ds has L_out / 2 rows (rounded down)
          store_h16(dsb + (size_t)(o >> 1) * COUT + cg * 16, v);
        }
      }
    }
    __syncthreads();
    if (tid < COUT) {
      // channel tid lives in units (j, cg = tid / 16), j = 0..MT-1; each unit was reduced by 4 warps (quads).
      float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
      for (int j = 0; j < MT; ++j) {
        const int unit = j * (COUT / 16) + (tid >> 4);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int slot = (((unit & 1) * 4 + q) * 4 + (unit >> 1)) * 16 + (tid & 15);
          s0 += sPartSum[slot];
          s1 += sPartSq[slot];
        }
      }
      // fp64 atomics: the cross-CTA summation order no longer changes the fp32 result (run-to-run determinism)
      atomicAdd(&p.out_stats[((size_t)b * COUT + tid) * 2 + 0], (double)s0);
      atomicAdd(&p.out_stats[((size_t)b * COUT + tid) * 2 + 1], (double)s1);
    }
  } else if (EPI == EPI_ACT_BWD) {
    constexpr int UNITS = MT * (COUT / 16);  // == 8
#pragma unroll 1
    for (int unit = wg; unit < UNITS; unit += 2) {
      const int j = unit / (COUT / 16);
      const int cg = unit % (COUT / 16);
      float v[16], gx[16];
      tmem_ld16(tmem_base + t_lane + j * COUT + cg * 16, v);
      const int o = o0 + j * 128 + quad * 32 + lane;
      const bool valid = o < p.L_out;
      if (valid) {
        const size_t off = ((size_t)b * p.L_out + o) * COUT + cg * 16;
        auto load16 = [&](const act_t* src, float* dst) {
          const uint4* q = reinterpret_cast<const uint4*>(src + off);
          const uint4 z[2] = {__ldg(q), __ldg(q + 1)};
          const uint32_t* w = reinterpret_cast<const uint32_t*>(z);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float2 f = unpack_h2(w[k]);
            dst[2 * k] = f.x;
            dst[2 * k + 1] = f.y;
          }
        };
        float y[16], r[16], act[16];
        load16(p.ab_y, y);
        if (p.res != nullptr) {  // second gradient contribution (1x1 stride-2 residual branch of the consumer block)
          load16(p.res, r);
#pragma unroll
          for (int k = 0; k < 16; ++k) v[k] += r[k];
        }
        if (p.ab_r != nullptr) load16(p.ab_r, r);
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const float xh = (y[k] - sShift[cg * 16 + k]) * sScale[cg * 16 + k];
          float g = v[k], a, da;
          gelu_tanh_both(xh, a, da);
          if (p.ab_r != nullptr) {
            float ds;
            gelu_tanh_both(a + r[k], a, ds);
            g *= ds;
            r[k] = g;  // dr
          }
          g *= da;
          v[k] = g;
          gx[k] = g * xh;
          act[k] = a;
        }
        store_h16(p.out + off, v);
        if (p.ab_a != nullptr) store_h16(p.ab_a + off, act);
        if (p.ab_r != nullptr) store_h16(p.ab_dr + off, r);
      } else {
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = gx[k] = 0.0f;
      }
      butterfly16(v, lane);
      butterfly16(gx, lane);
      if ((lane & 1) == 0) {
        const int slot = (warp * 4 + (unit >> 1)) * 16 + butterfly16_channel(lane);
        sPartSum[slot] = v[0];
        sPartSq[slot] = gx[0];
      }
    }
    __syncthreads();
    if (tid < COUT) {
      float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
      for (int j = 0; j < MT; ++j) {
        const int unit = j * (COUT / 16) + (tid >> 4);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int slot = (((unit & 1) * 4 + q) * 4 + (unit >> 1)) * 16 + (tid & 15);
          s0 += sPartSum[slot];
          s1 += sPartSq[slot];
        }
      }
      atomicAdd(&p.out_stats[((size_t)b * COUT + tid) * 2 + 0], (double)s0);
      atomicAdd(&p.out_stats[((size_t)b * COUT + tid) * 2 + 1], (double)s1);
    }
  } else if (EPI == EPI_PLAIN) {
    constexpr int UNITS = MT * (COUT / 16);
#pragma unroll 1
    for (int unit = wg; unit < UNITS; unit += 2) {
      const int j = unit / (COUT / 16);
      const int cg = unit % (COUT / 16);
      float v[16];
      tmem_ld16(tmem_base + t_lane + j * COUT + cg * 16, v);
      const int o = o0 + j * 128 + quad * 32 + lane;
      if (o < p.L_out) {
        const size_t off = ((size_t)b * p.out_rows + (size_t)o * p.out_stride + p.out_offset) * COUT + cg * 16;
        if (p.bias != nullptr) {
#pragma unroll
          for (int k = 0; k < 16; ++k) v[k] += __ldg(p.bias + cg * 16 + k);
        }
        if (p.res != nullptr) {
          const uint4* rp = reinterpret_cast<const uint4*>(p.res + off);
          uint4 rz[2] = {__ldg(rp), __ldg(rp + 1)};
          const uint32_t* rr = reinterpret_cast<const uint32_t*>(rz);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float2 r2 = unpack_h2(rr[k]);
            v[2 * k] += r2.x;
            v[2 * k + 1] += r2.y;
          }
        }
        store_h16(p.out + off, v);
      }
    }
  } else if (EPI == EPI_BIAS_GELU) {
    act_t* outb = p.out + (size_t)b * p.L_out * COUT;
    const int o = o0 + quad * 32 + lane;
#pragma unroll 1
    for (int cg = wg; cg < COUT / 16; cg += 2) {
      float v[16];
      tmem_ld16(tmem_base + t_lane + cg * 16, v);
      if (o < p.L_out) {
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = gelu_erf(v[k] + __ldg(p.bias + cg * 16 + k));
        store_h16(outb + (size_t)o * COUT + cg * 16, v);
      }
    }
  } else {  // EPI_LN_GELU / EPI_LN_GELU_RES : thread owns one row of all 128 channels
    if (wg == 0) {
      const int o = o0 + quad * 32 + lane;
      const bool valid = o < p.L_out;
      // Three passes over TMEM (cheap) keep the two-pass variance of ConvLayerNorm (utils.py:17-21).
      float mean = 0.0f;
#pragma unroll 1
      for (int cg = 0; cg < 8; ++cg) {
        float v[16];
        tmem_ld16(tmem_base + t_lane + cg * 16, v);
#pragma unroll
        for (int k = 0; k < 16; ++k) mean += v[k];
      }
      mean *= (1.0f / 128.0f);
      float var = 0.0f;
#pragma unroll 1
      for (int cg = 0; cg < 8; ++cg) {
        float v[16];
        tmem_ld16(tmem_base + t_lane + cg * 16, v);
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const float d = v[k] - mean;
          var = fmaf(d, d, var);
        }
      }
      const float rstd = rsqrtf(var * (1.0f / 128.0f) + p.ln_eps);
      float lg[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) lg[c] = 0.0f;
      const size_t rowoff = ((size_t)b * p.L_out + (valid ? o : 0)) * COUT;
#pragma unroll 1
      for (int cg = 0; cg < 8; ++cg) {
        float v[16];
        tmem_ld16(tmem_base + t_lane + cg * 16, v);
        uint4 rz[2];
        if (EPI == EPI_LN_GELU_RES) {
          const uint4* rp = reinterpret_cast<const uint4*>(p.res + rowoff + cg * 16);
          rz[0] = __ldg(rp);
          rz[1] = __ldg(rp + 1);
        }
        const uint32_t* rr = reinterpret_cast<const uint32_t*>(rz);
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const int c = cg * 16 + k;
          float y = (v[k] - mean) * rstd * __ldg(p.ln_w + c) + __ldg(p.ln_b + c);
          y = gelu_erf(y);
          if (EPI == EPI_LN_GELU_RES) {
            const float2 r2 = unpack_h2(rr[k >> 1]);
            y = gelu_erf(y + ((k & 1) ? r2.y : r2.x));
          }
          v[k] = y;
        }
        if (EPI == EPI_LN_GELU_RES && p.head_w != nullptr) {
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            if (c < p.n_classes) {
              float acc = lg[c];
#pragma unroll
              for (int k = 0; k < 16; ++k) acc = fmaf(v[k], __ldg(p.head_w + c * COUT + cg * 16 + k), acc);
              lg[c] = acc;
            }
          }
        }
        if (valid) {
          store_h16(p.out + rowoff + cg * 16, v);
        }
      }
      if (EPI == EPI_LN_GELU_RES && p.head_w != nullptr && valid) {
        float* lrow = p.logits + ((size_t)b * p.L_out + o) * p.n_classes;
#pragma unroll
        for (int c = 0; c < 8; ++c)
          if (c < p.n_classes) lrow[c] = lg[c] + __ldg(p.head_b + c);
      }
    }
  }

  // ---------------- teardown ----------------
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, TMEM_COLS);
}

template <int CIN, int COUT, int TAPS, int GT, int PRO, int EPI, bool HAS_DS, bool SPLIT, bool BF16OP = false>
__global__ void __launch_bounds__(kConvThreads, (EPI == EPI_ACT_BWD && COUT <= 64) ? 3 : 1) conv_igemm_kernel(const ConvArgs p) {
  conv_igemm_body<CIN, COUT, TAPS, GT, PRO, EPI, HAS_DS, SPLIT, BF16OP>(p, (int)blockIdx.y);
}
// The same tile program for two argument sets in one grid (blockIdx.z selects): the encoder Linear of two encoders of
// identical architecture (w2s_encoder_fwd_pair).  Instantiated for those configurations only.
template <int CIN, int COUT, int TAPS, int GT, int PRO, int EPI, bool HAS_DS, bool SPLIT>
__global__ void __launch_bounds__(kConvThreads, 1) conv_igemm_pair_kernel(const ConvArgs pa, const ConvArgs pb) {
  // two copies of the tile program, each reading its own argument block straight from the parameter space (selecting
  // single pointers into a local ConvArgs instead lost the override of `in` in the generated code: the second
  // encoder's Linear read the first encoder's activations - caught by the paired-vs-single parity test)
  if (blockIdx.z != 0) conv_igemm_body<CIN, COUT, TAPS, GT, PRO, EPI, HAS_DS, SPLIT, false>(pb, (int)blockIdx.y);
  else conv_igemm_body<CIN, COUT, TAPS, GT, PRO, EPI, HAS_DS, SPLIT, false>(pa, (int)blockIdx.y);
}

template <int CIN, int COUT, int TAPS, int GT, int PRO, int EPI, bool HAS_DS>
inline cudaError_t launch_conv_igemm_pair(const ConvArgs& a, const ConvArgs& a2, int B, cudaStream_t stream) {
  constexpr bool SPLIT = ConvSplit<CIN, COUT>::value && EPI == EPI_STATS;
  auto kern = conv_igemm_pair_kernel<CIN, COUT, TAPS, GT, PRO, EPI, HAS_DS, SPLIT>;
  const int stride = 1 << a.stride_log2;
  const size_t smem = conv_smem_bytes<CIN, COUT, GT, HAS_DS, SPLIT>(stride, TAPS, a.dil);
  static size_t configured = 0;  // per instantiation
  if (smem > configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    configured = smem;
  }
  dim3 grid((a.L_out + ConvTile<COUT>::POS - 1) / ConvTile<COUT>::POS, B, 2);
  kern<<<grid, kConvThreads, smem, stream>>>(a, a2);
  return cudaGetLastError();
}

// Dynamic shared memory of one launch_conv_igemm call.
template <int CIN, int COUT, int TAPS, int GT, int EPI, bool HAS_DS, bool BF16OP = false>
inline size_t conv_igemm_smem_bytes(const ConvArgs& a) {
  constexpr bool SPLIT = ConvSplit<CIN, COUT>::value && EPI == EPI_STATS && !BF16OP;
  return conv_smem_bytes<CIN, COUT, GT, HAS_DS, SPLIT>(1 << a.stride_log2, TAPS, a.dil);
}

// Host-side launcher.  Returns cudaError_t of the launch.
template <int CIN, int COUT, int TAPS, int GT, int PRO, int EPI, bool HAS_DS, bool BF16OP = false>
inline cudaError_t launch_conv_igemm(const ConvArgs& a, int B, cudaStream_t stream) {
  constexpr bool SPLIT = ConvSplit<CIN, COUT>::value && EPI == EPI_STATS && !BF16OP;
  auto kern = conv_igemm_kernel<CIN, COUT, TAPS, GT, PRO, EPI, HAS_DS, SPLIT, BF16OP>;
  const size_t smem = conv_igemm_smem_bytes<CIN, COUT, TAPS, GT, EPI, HAS_DS, BF16OP>(a);
  static size_t configured = 0;  // per instantiation
  if (smem > configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    configured = smem;
  }
  dim3 grid((a.L_out + ConvTile<COUT>::POS - 1) / ConvTile<COUT>::POS, B);
  kern<<<grid, kConvThreads, smem, stream>>>(a);
  return cudaGetLastError();
}

}  // namespace w2s
