// C ABI of libw2s_b200 (see include/w2s_b200.h).  Host-side orchestration only: shape checks, workspace
// carving, kernel dispatch.  No allocation, no synchronisation, no CPU fallback.
#include "../../include/w2s_b200.h"

#include <cuda_bf16.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cmath>
#include <cstring>
#include <cstdlib>
#include <mutex>
#include <string>
#include <vector>

#include "attribution.cuh"
#include "conv_igemm.cuh"
#include "conv_stream.cuh"
#include "epoch_mixer.cuh"
#include "first_conv.cuh"
#include "gemm_tn.cuh"
#include "train_kernels.cuh"
#include "general.cuh"
#include "general_bwd.cuh"
#include "staging.cuh"
#include "seq_mixer.cuh"
#include "stream.cuh"

using namespace w2s;

namespace {

thread_local std::string g_err;

int fail(const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return 1;
}
int cuda_fail(cudaError_t e, const char* what) { return fail("%s: %s", what, cudaGetErrorString(e)); }

int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ------------------------------------------------------------------------------------------------
// launch accounting + optional per-launch CUDA-event profile (bench.py reads it; off by default)
// ------------------------------------------------------------------------------------------------
std::atomic<long long> g_launches{0};
std::atomic<int> g_conv_impl{0};  // 0 = auto (persistent streaming kernel where built), 1 = tile-per-CTA kernel only
struct ProfRec {
  std::string label;
  cudaEvent_t e0, e1;
  double bytes, flops;
};
std::mutex g_prof_mu;
bool g_prof_on = false;
std::vector<ProfRec> g_prof;

// RAII around one kernel launch: counts it and, when profiling, brackets it with events on its stream.
struct LaunchScope {
  cudaStream_t st;
  bool on;
  size_t idx;
  LaunchScope(cudaStream_t s, const char* label, double bytes, double flops) : st(s), on(false), idx(0) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (!g_prof_on) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    ProfRec r;
    r.label = label;
    r.bytes = bytes;
    r.flops = flops;
    if (cudaEventCreate(&r.e0) != cudaSuccess || cudaEventCreate(&r.e1) != cudaSuccess) return;
    cudaEventRecord(r.e0, st);
    g_prof.push_back(r);
    idx = g_prof.size() - 1;
    on = true;
  }
  ~LaunchScope() {
    if (!on) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    cudaEventRecord(g_prof[idx].e1, st);
  }
};

// ------------------------------------------------------------------------------------------------
// packing kernels
// ------------------------------------------------------------------------------------------------
__global__ void pack_conv_kernel(const float* __restrict__ w, int cout, int cin, int taps, int taps_major, int split,
                                 __half* __restrict__ out) {
  const int total = taps * cin * cout;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int k = idx & 7;
    int r = idx >> 3;
    const int n = r % cout;
    r /= cout;
    const int c8 = r % (cin / 8);
    const int t = r / (cin / 8);
    const int c = c8 * 8 + k;
    const float v = taps_major ? w[(size_t)n * taps * cin + (size_t)t * cin + c] : w[((size_t)n * cin + c) * taps + t];
    if (split == 2) {  // bf16 operand (measurement hook): one block of bf16 bit patterns
      reinterpret_cast<__nv_bfloat16*>(out)[idx] = __float2bfloat16_rn(v);
      continue;
    }
    const __half hi = __float2half_rn(v);
    out[idx] = hi;
    if (split) out[total + idx] = __float2half_rn(v - __half2float(hi));  // W = hi + lo
  }
}

// All weight re-packing of a model in ONE launch (after every optimizer step): blockIdx.y = job.  A job reads its source
// through explicit element strides (so flipped / transposed / sliced views of the fp32 master parameters need no torch
// copies) and writes either the UMMA conv layout (kind 0, optionally hi + lo) or the mma.sync fragment order (kind 1).
__global__ void pack_batch_kernel(const w2s_pack_job* __restrict__ jobs) {
  const w2s_pack_job j = jobs[blockIdx.y];
  __half* out = reinterpret_cast<__half*>(j.out);
  if (j.kind == 0) {
    const int cout = j.cout, cin = j.cin, taps = j.taps;
    const int total = taps * cin * cout;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
      const int k = idx & 7;
      int r = idx >> 3;
      const int n = r % cout;
      r /= cout;
      const int c8 = r % (cin / 8);
      const int t = r / (cin / 8);
      const int c = c8 * 8 + k;
      const float v = j.w[(long long)n * j.sn + (long long)c * j.sc + (long long)t * j.st];
      const __half hi = __float2half_rn(v);
      out[idx] = hi;
      if (j.split) out[total + idx] = __float2half_rn(v - __half2float(hi));
    }
  } else {  // nn.Linear weight [n, k] (row stride sn, column stride sc) -> mma.sync B-fragment order
    const int n_ = j.cout, k_ = j.cin;
    const int total = n_ * k_;
    const int KT = k_ / 16;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
      const int q = idx & 3;
      const int lane = (idx >> 2) & 31;
      const int tile = idx >> 7;
      const int kt = tile % KT, nt = tile / KT;
      const int row = nt * 8 + (lane >> 2);
      const int col = kt * 16 + (lane & 3) * 2 + (q & 1) + (q >> 1) * 8;
      out[idx] = __float2half_rn(j.w[(long long)row * j.sn + (long long)col * j.sc]);
    }
  }
}

__global__ void pack_frag_kernel(const float* __restrict__ w, int n, int k, __half* __restrict__ out) {
  const int total = n * k;
  const int KT = k / 16;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int q = idx & 3;
    const int lane = (idx >> 2) & 31;
    const int tile = idx >> 7;
    const int kt = tile % KT, nt = tile / KT;
    const int row = nt * 8 + (lane >> 2);
    const int col = kt * 16 + (q >> 1) * 8 + (lane & 3) * 2 + (q & 1);
    out[idx] = __float2half_rn(w[(size_t)row * k + col]);
  }
}

__global__ void argmax_kernel(const float* __restrict__ logits, long long n, int c, long long* __restrict__ out) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float* row = logits + i * c;
    int best = 0;
    float bv = row[0];
    for (int j = 1; j < c; ++j) {
      const float v = row[j];
      if (v > bv) {  // first maximum wins, like torch.argmax
        bv = v;
        best = j;
      }
    }
    out[i] = best;
  }
}

// ------------------------------------------------------------------------------------------------
// generic conv dispatch
// ------------------------------------------------------------------------------------------------
int ilog2_exact(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return (1 << l) == v ? l : -1;
}

ConvArgs to_args(const w2s_conv_call& c) {
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.in = (const act_t*)c.in;
  a.in_res = (const act_t*)c.in_res;
  a.in_stats = c.in_stats;
  a.w = (const act_t*)c.w;
  a.w_ds = (const act_t*)c.w_ds;
  a.out = (act_t*)c.out;
  a.out_ds = (act_t*)c.out_ds;
  a.out_stats = c.out_stats;
  a.row_mask = c.row_mask;
  a.bias = c.bias;
  a.ln_w = c.ln_w;
  a.ln_b = c.ln_b;
  a.res = (const act_t*)c.res;
  a.head_w = c.head_w;
  a.head_b = c.head_b;
  a.logits = c.logits;
  a.n_classes = c.n_classes;
  a.L_in = c.L_in;
  a.L_out = c.L_out;
  a.stride_log2 = ilog2_exact(c.stride);
  a.dil = c.dilation;
  a.pad = c.pad;
  a.in_eps = c.in_eps;
  a.ln_eps = c.ln_eps;
  a.x_raw = c.x_raw; a.w_first = c.w_first; a.w_first_ds = c.w_first_ds; a.T_raw = c.T_raw;
  a.out_stride = c.out_stride > 0 ? c.out_stride : 1;
  a.out_offset = c.out_offset;
  a.out_rows = c.out_rows > 0 ? c.out_rows : c.L_out;
  a.ab_y = (const act_t*)c.act_y; a.ab_r = (const act_t*)c.act_r; a.ab_stats = c.act_stats;
  a.ab_a = (act_t*)c.act_a; a.ab_dr = (act_t*)c.act_dr; a.ab_eps = c.act_eps;
  a.dn_sums = c.dn_sums; a.dn_out = (act_t*)c.dn_out; a.dn_upsample = c.dn_upsample;
  { const char* dbg = getenv("W2S_DEBUG_FLAGS"); a.debug_flags = dbg ? atoi(dbg) : 0; }
  return a;
}

// c2 != nullptr: a second call of the same shape and configuration (the same layer of a second encoder with identical
// architecture) to run in the same launch (paired stream kernel, conv_stream.cuh).  Returns kNotPaired - nothing was
// launched - if the pair cannot share a launch; the caller then dispatches the two calls one after the other.
constexpr int kNotPaired = -77;
static bool conv_calls_pairable(const w2s_conv_call& a, const w2s_conv_call& b) {
  return a.cin == b.cin && a.cout == b.cout && a.taps == b.taps && a.stride == b.stride && a.dilation == b.dilation &&
         a.pad == b.pad && a.prologue == b.prologue && a.epilogue == b.epilogue && a.has_ds == b.has_ds && a.B == b.B &&
         a.L_in == b.L_in && a.L_out == b.L_out && a.in_wide == b.in_wide && a.out_wide == b.out_wide &&
         a.force_split == b.force_split && a.T_raw == b.T_raw && a.in_eps == b.in_eps &&
         (a.row_mask != nullptr) == (b.row_mask != nullptr) && (a.bias != nullptr) == (b.bias != nullptr);
}

// Shared memory one block may opt in to on this device (232,448 B on sm_100).
int smem_optin_bytes() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (n <= 0) n = 232448;
  }
  return n;
}

// The tile-per-CTA kernel stages every input row its 128-position tile reaches, (taps - 1) * dilation of them beyond
// the tile, so a wide dilation can need more shared memory than a block can have (k7 128 -> 128: 220,176 B at dilation
// 32, 269,328 B at 64).  Such a call fails with its layer shape and byte count instead of the bare attribute error.
template <int CIN, int COUT, int TAPS, int GT, int PRO, int EPI, bool DS, bool BF16OP = false>
int run_conv_igemm(const w2s_conv_call& c, const ConvArgs& a, cudaStream_t st) {
  const size_t smem = conv_igemm_smem_bytes<CIN, COUT, TAPS, GT, EPI, DS, BF16OP>(a);
  if (smem > (size_t)smem_optin_bytes())
    return fail("conv1d: c%d->%d k%d stride %d dilation %d needs %zu B of shared memory per block, over the %d B limit "
                "of this device", c.cin, c.cout, c.taps, c.stride, c.dilation, smem, smem_optin_bytes());
  const cudaError_t e = launch_conv_igemm<CIN, COUT, TAPS, GT, PRO, EPI, DS, BF16OP>(a, c.B, st);
  return e == cudaSuccess ? 0 : cuda_fail(e, "conv1d launch");
}

int conv_dispatch(const w2s_conv_call& c, cudaStream_t st, const w2s_conv_call* c2 = nullptr) {
  if (c2 != nullptr && !conv_calls_pairable(c, *c2)) return kNotPaired;
  if (c.B <= 0 || c.L_in <= 0 || c.L_out <= 0) return fail("conv1d: empty shape B=%d L_in=%d L_out=%d", c.B, c.L_in, c.L_out);
  if (ilog2_exact(c.stride) < 0 || c.stride > 4) return fail("conv1d: stride %d unsupported", c.stride);
  if (c.B > 65535) return fail("conv1d: B=%d exceeds grid.y", c.B);
  if (c.n_classes > 8) return fail("conv1d: n_classes=%d > 8", c.n_classes);
  const int impl = g_conv_impl.load();
  if ((c.in_wide || c.out_wide || c.force_split) && (c.epilogue != W2S_EPI_STATS || impl != 0))
    return fail("conv1d: wide storage / forced split operands are only built for the streaming encoder kernels");
  if (c.prologue == W2S_PRO_DNORM) {
    if (c.epilogue != W2S_EPI_ACT_BWD || c.stride != 1 || c.taps != 3 || c.L_in != c.L_out)
      return fail("conv1d: W2S_PRO_DNORM is built for the k3 stride-1 data-gradient convs (W2S_EPI_ACT_BWD) only");
    if (!c.in_res || !c.in_stats || !c.dn_sums || !c.dn_out) return fail("conv1d: W2S_PRO_DNORM needs in_res (y), in_stats, dn_sums, dn_out");
    if (c.dn_upsample && (c.L_in & 1)) return fail("conv1d: W2S_PRO_DNORM upsample needs an even L_in");
  }
  // the block-0 fusion kernels stage each night's raw-signal window with 16-byte bulk copies from x_raw + b * T_raw
  // (both calls of a pair: conv_calls_pairable compares T_raw but not the pointers)
  for (const w2s_conv_call* q : {&c, c2}) {
    if (q == nullptr || (q->prologue != W2S_PRO_FIR && q->prologue != W2S_PRO_NORM_RES_X)) continue;
    if (q->x_raw == nullptr || q->T_raw <= 0 || (q->T_raw & 3))
      return fail("conv1d: W2S_PRO_FIR / W2S_PRO_NORM_RES_X need x_raw and a T_raw that is a multiple of 4 (got x_raw=%p "
                  "T_raw=%d, L_in=%d)", (const void*)q->x_raw, q->T_raw, q->L_in);
  }
  if (c.epilogue == W2S_EPI_ACT_BWD) {
    if (!c.act_y || !c.act_stats || !c.out_stats || (c.act_r && !c.act_dr))
      return fail("conv1d: W2S_EPI_ACT_BWD needs act_y, act_stats, out_stats (and act_dr with act_r)");
    if (c.out_stride > 1 || c.out_offset != 0 || (c.out_rows > 0 && c.out_rows != c.L_out))
      return fail("conv1d: W2S_EPI_ACT_BWD writes dense rows only");
  }
  if (c.epilogue == W2S_EPI_PLAIN) {  // output row o * out_stride + out_offset of a sample of out_rows rows
    const int os = c.out_stride > 0 ? c.out_stride : 1, rows = c.out_rows > 0 ? c.out_rows : c.L_out;
    if (c.out_offset < 0 || c.out_offset >= os || (long long)(c.L_out - 1) * os + c.out_offset >= rows)
      return fail("conv1d: W2S_EPI_PLAIN output rows out of range: L_out=%d out_stride=%d out_offset=%d out_rows=%d "
                  "(needs 0 <= out_offset < out_stride and (L_out - 1) * out_stride + out_offset < out_rows)",
                  c.L_out, os, c.out_offset, rows);
  }
  const ConvArgs a = to_args(c);
  ConvArgs a2s;
  const ConvArgs* a2 = nullptr;
  if (c2 != nullptr) {
    a2s = to_args(*c2);
    a2 = &a2s;
  }
  const double npair = c2 != nullptr ? 2.0 : 1.0;
  cudaError_t e = cudaErrorInvalidValue;
  bool found = false;
  char label[96];
  snprintf(label, sizeof(label), "conv c%d->%d k%d s%d d%d pro%d epi%d%s%s%s B%d L%d", c.cin, c.cout, c.taps, c.stride,
           c.dilation, c.prologue, c.epilogue, c.has_ds ? " +ds" : "",
           c.in_wide ? (c.out_wide ? " w32/32" : " w32/16") : (c.out_wide ? " w16/32" : ""),
           c2 != nullptr ? " x2" : "", c.B, c.L_in);  // x2: paired launch (two encoders, B nights each)
  const double ein = c.in_wide ? 4.0 : 2.0, eout = c.out_wide ? 4.0 : 2.0;
  // algorithmic traffic: every input element read once (+ residual), every output written once; fp16
  const double in_b = c.prologue == W2S_PRO_DNORM  // d(x_hat) + y read (half length when zero-stuffed), dy written
                          ? (double)c.B * c.L_in * c.cin * 2.0 * (c.dn_upsample ? 2.0 : 3.0)
                      : c.prologue == W2S_PRO_FIR ? (double)c.B * c.L_in * 4.0
                      : (double)c.B * c.L_in * c.cin * ein * (c.prologue == W2S_PRO_NORM_RES ? 2.0 : 1.0) +
                            (c.prologue == W2S_PRO_NORM_RES_X ? (double)c.B * c.L_in * 8.0 : 0.0);
  const double out_b = (double)c.B * c.L_out * c.cout * eout * (c.has_ds ? 1.5 : 1.0) +
                       (c.epilogue == W2S_EPI_LN_GELU_RES ? (double)c.B * c.L_out * c.cout * 2.0 : 0.0);
  const double ab_b = c.epilogue == W2S_EPI_ACT_BWD
                          ? (double)c.B * c.L_out * c.cout * 2.0 * (1.0 + (c.res ? 1.0 : 0.0) + (c.act_r ? 2.0 : 0.0) + (c.act_a ? 1.0 : 0.0))
                          : 0.0;
  const double fl = 2.0 * c.B * (double)c.L_out * c.cout * c.cin * (c.taps + (c.has_ds ? 0.5 : 0.0));
  // a pair whose shape has no stream kernel is not launched here (checked before the launch is counted / timed)
  const bool stream_shape = c.epilogue == W2S_EPI_STATS && c.taps == 3 && c.dilation == 1 && c.pad == 1 && impl == 0 &&
                            ((c.stride == 1 && c.L_out == c.L_in) || (c.stride == 2 && c.L_out == (c.L_in + 1) / 2));
  // the encoder Linear (4-tap stride-4 conv + bias + GELU, tile-per-CTA kernel): paired through blockIdx.z
  const bool linear_shape = c.epilogue == W2S_EPI_BIAS_GELU && c.taps == 4 && c.stride == 4 && c.dilation == 1 && c.pad == 0 &&
                            c.prologue == W2S_PRO_NORM_RES && !c.has_ds && impl == 0 && c.cout == 128 &&
                            (c.cin == 64 || c.cin == 128) && !c.in_wide && !c.out_wide && !c.force_split;
  if (c2 != nullptr && !((stream_shape && stream_pairable(c.cout, c.has_ds != 0)) || linear_shape))
    return kNotPaired;
  LaunchScope scope(st, label, npair * (in_b + out_b + ab_b), npair * fl);
  if (stream_shape) {
    const int sms = sm_count();
    const bool want_split = c.force_split != 0 || w2s_conv_uses_split(c.cin, c.cout) != 0;
#define W2S_STREAMX(CIN, COUT, STRIDE, PRO, DS, MT, NR, NA, NTW, WIN, WOUT, SPLIT)                          \
  if (!found && c.cin == CIN && c.cout == COUT && c.stride == STRIDE && c.prologue == PRO && (c.has_ds != 0) == DS && \
      (c.in_wide != 0) == WIN && (c.out_wide != 0) == WOUT && want_split == SPLIT) {                        \
    found = true;                                                                                           \
    e = launch_conv_stream<CIN, COUT, STRIDE, PRO, DS, MT, NR, NA, NTW, WIN, WOUT, SPLIT>(a, a2, c.B, sms, st); \
  }
#define W2S_STREAMW(CIN, COUT, STRIDE, PRO, DS, MT, NR, NA, NTW, WIN, WOUT) \
  W2S_STREAMX(CIN, COUT, STRIDE, PRO, DS, MT, NR, NA, NTW, WIN, WOUT, (CIN <= 16 && COUT <= 16))
#define W2S_STREAM(CIN, COUT, STRIDE, PRO, DS, MT, NR, NA, NTW) \
  W2S_STREAMW(CIN, COUT, STRIDE, PRO, DS, MT, NR, NA, NTW, false, false)
    //          cin cout s  prologue      ds    MT NR NA NTW
    W2S_STREAM(16, 16, 1, PRO_FIR, false, 8, 3, 2, 18)
    W2S_STREAM(16, 16, 1, PRO_NORM_RES_X, true, 8, 2, 2, 14)
    W2S_STREAM(16, 16, 1, PRO_NORM, false, 8, 2, 2, 18)
    W2S_STREAM(16, 16, 2, PRO_NORM, false, 4, 2, 2, 18)
    W2S_STREAM(16, 16, 1, PRO_NORM_RES, true, 4, 3, 2, 14)
    // (10 transform warps at 120 registers; 12 / 14 warps cap the kernel at 96 registers and spill: 16 -> 32 conv1
    //  265 -> 339 / 361 us per paired launch, 32 -> 32 conv1 227 -> 214 / 241 us, step +2-3 %)
    W2S_STREAM(16, 32, 1, PRO_NORM_RES, true, 4, 3, 2, 10)
    W2S_STREAM(32, 32, 1, PRO_NORM, false, 4, 2, 2, 14)
    W2S_STREAM(32, 32, 2, PRO_NORM, false, 2, 2, 2, 14)
    W2S_STREAM(32, 32, 1, PRO_NORM_RES, true, 2, 3, 2, 10)
    W2S_STREAM(32, 64, 1, PRO_NORM_RES, true, 2, 3, 2, 14)
    W2S_STREAM(64, 64, 1, PRO_NORM, false, 2, 2, 2, 14)
    W2S_STREAM(64, 64, 2, PRO_NORM, false, 1, 3, 2, 14)
    W2S_STREAM(64, 64, 1, PRO_NORM_RES, true, 1, 3, 2, 14)
    W2S_STREAM(64, 128, 1, PRO_NORM_RES, true, 1, 0, 3, 14)  // direct: 68 vs 75 us (the 64 -> 64 kernels lose 12-20 %)
    // NR = 0 (direct from global, conv_stream.cuh): the 128-channel weights leave room for one A stage next to a raw
    // ring, and two or three without one
    W2S_STREAM(128, 128, 1, PRO_NORM, false, 1, 0, 3, 14)
    W2S_STREAM(128, 128, 2, PRO_NORM, false, 1, 0, 2, 14)
    W2S_STREAM(128, 128, 1, PRO_NORM_RES, true, 1, 0, 2, 14)
    // wide (fp32) storage of the leading <= 32-channel blocks            MT NR NA NTW  in     out
    W2S_STREAMW(16, 16, 1, PRO_FIR, false, 8, 3, 2, 18, false, true)
    W2S_STREAMW(16, 16, 1, PRO_NORM_RES_X, true, 4, 3, 2, 14, true, true)
    W2S_STREAMW(16, 16, 1, PRO_NORM, false, 6, 2, 2, 18, true, true)
    W2S_STREAMW(16, 16, 2, PRO_NORM, false, 3, 2, 2, 18, true, true)
    W2S_STREAMX(16, 32, 1, PRO_NORM_RES, true, 4, 2, 2, 10, true, false, false)
    W2S_STREAMX(16, 32, 1, PRO_NORM_RES, true, 4, 2, 2, 10, true, true, true)
    W2S_STREAMX(32, 32, 1, PRO_NORM, false, 3, 2, 2, 14, true, true, true)
    W2S_STREAMX(32, 32, 2, PRO_NORM, false, 1, 3, 2, 14, true, true, true)
    W2S_STREAMX(32, 32, 1, PRO_NORM_RES, true, 2, 2, 2, 10, true, true, true)
    W2S_STREAMX(32, 64, 1, PRO_NORM_RES, true, 2, 2, 2, 14, true, false, false)
    // wide storage + split operands of the 64-channel blocks (wide_blocks = 6: >= 10-block encoders, DESIGN.md "Numerics")
    //                                                 MT NR NA NTW  in    out   split
    W2S_STREAMX(32, 64, 1, PRO_NORM_RES, true, 2, 1, 2, 14, true, true, true)
    W2S_STREAMX(64, 64, 1, PRO_NORM, false, 1, 2, 2, 14, true, true, true)
    W2S_STREAMX(64, 64, 2, PRO_NORM, false, 1, 1, 1, 14, true, true, true)
    W2S_STREAMX(64, 64, 1, PRO_NORM_RES, true, 1, 1, 2, 14, true, true, true)
    W2S_STREAMX(64, 128, 1, PRO_NORM_RES, true, 1, 1, 2, 14, true, false, false)
#undef W2S_STREAM
#undef W2S_STREAMW
#undef W2S_STREAMX
    if (!found && (c.in_wide || c.out_wide || c.force_split))
      return fail("conv1d: no wide-storage kernel for cin=%d cout=%d stride=%d prologue=%d in_wide=%d out_wide=%d split=%d",
                  c.cin, c.cout, c.stride, c.prologue, c.in_wide, c.out_wide, (int)want_split);
    if (found) {
      if (e != cudaSuccess) return cuda_fail(e, "conv_stream launch");
      return 0;
    }
  }
  if (c2 != nullptr && linear_shape) {
    e = c.cin == 64 ? launch_conv_igemm_pair<64, 128, 4, 4, PRO_NORM_RES, EPI_BIAS_GELU, false>(a, a2s, c.B, st)
                    : launch_conv_igemm_pair<128, 128, 4, 2, PRO_NORM_RES, EPI_BIAS_GELU, false>(a, a2s, c.B, st);
    return e == cudaSuccess ? 0 : cuda_fail(e, "conv_igemm pair launch");
  }
  if (c2 != nullptr) return kNotPaired;  // no stream kernel for this configuration: the caller dispatches the two calls singly
  if (impl == 3) {  // bf16 operands on the tile-per-CTA kernel: un-split encoder convs without the 1x1 branch only
#define W2S_BF16(CIN, COUT)                                                                                          \
  if (c.cin == CIN && c.cout == COUT && c.taps == 3 && c.prologue == PRO_NORM && c.epilogue == EPI_STATS && !c.has_ds) \
    return run_conv_igemm<CIN, COUT, 3, 3, PRO_NORM, EPI_STATS, false, true>(c, a, st);
    W2S_BF16(32, 32)
    W2S_BF16(64, 64)
    W2S_BF16(128, 128)
#undef W2S_BF16
    return fail("conv1d: bf16-operand hook is built for k3 32->32 / 64->64 / 128->128 EPI_STATS convs only");
  }
#define W2S_CASE(CIN, COUT, TAPS, GT, PRO, EPI, DS)                                                                  \
  if (c.cin == CIN && c.cout == COUT && c.taps == TAPS && c.prologue == PRO && c.epilogue == EPI && (c.has_ds != 0) == DS) \
    return run_conv_igemm<CIN, COUT, TAPS, GT, PRO, EPI, DS>(c, a, st);
  // encoder conv1 (block input = previous block's conv3 output + residual branch), with fused downsample
  W2S_CASE(16, 16, 3, 3, PRO_NORM_RES, EPI_STATS, true)
  W2S_CASE(16, 32, 3, 3, PRO_NORM_RES, EPI_STATS, true)
  W2S_CASE(32, 32, 3, 3, PRO_NORM_RES, EPI_STATS, true)
  W2S_CASE(32, 64, 3, 3, PRO_NORM_RES, EPI_STATS, true)
  W2S_CASE(64, 64, 3, 3, PRO_NORM_RES, EPI_STATS, true)
  W2S_CASE(64, 128, 3, 3, PRO_NORM_RES, EPI_STATS, true)
  W2S_CASE(128, 128, 3, 3, PRO_NORM_RES, EPI_STATS, true)
  // encoder conv2 / conv3 (stride is a runtime argument)
  W2S_CASE(16, 16, 3, 3, PRO_NORM, EPI_STATS, false)
  W2S_CASE(32, 32, 3, 3, PRO_NORM, EPI_STATS, false)
  W2S_CASE(64, 64, 3, 3, PRO_NORM, EPI_STATS, false)
  W2S_CASE(128, 128, 3, 3, PRO_NORM, EPI_STATS, false)
  // encoder Linear(4C -> 128) + GELU as a 4-tap stride-4 conv
  W2S_CASE(64, 128, 4, 4, PRO_NORM_RES, EPI_BIAS_GELU, false)
  W2S_CASE(128, 128, 4, 2, PRO_NORM_RES, EPI_BIAS_GELU, false)
  // sequence mixer dilated convs
  W2S_CASE(128, 128, 7, 4, PRO_NONE, EPI_LN_GELU, false)
  W2S_CASE(128, 128, 7, 4, PRO_NONE, EPI_LN_GELU_RES, false)
  // training path: plain GEMMs (taps 1 / 4) and data-gradient convolutions (input already materialised)
  W2S_CASE(128, 128, 1, 1, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(128, 128, 4, 2, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(64, 128, 4, 4, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(128, 128, 7, 4, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(128, 64, 1, 1, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(16, 16, 3, 3, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(32, 16, 3, 3, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(32, 32, 3, 3, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(64, 32, 3, 3, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(64, 64, 3, 3, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(128, 64, 3, 3, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(128, 128, 3, 3, PRO_NONE, EPI_PLAIN, false)
  // training: data-gradient convs fused with the activation backward of the producing layer
  W2S_CASE(16, 16, 3, 3, PRO_NONE, EPI_ACT_BWD, false)
  W2S_CASE(32, 16, 3, 3, PRO_NONE, EPI_ACT_BWD, false)
  W2S_CASE(32, 32, 3, 3, PRO_NONE, EPI_ACT_BWD, false)
  W2S_CASE(64, 32, 3, 3, PRO_NONE, EPI_ACT_BWD, false)
  W2S_CASE(64, 64, 3, 3, PRO_NONE, EPI_ACT_BWD, false)
  W2S_CASE(128, 64, 3, 3, PRO_NONE, EPI_ACT_BWD, false)
  W2S_CASE(128, 128, 3, 3, PRO_NONE, EPI_ACT_BWD, false)
  // ... with the InstanceNorm backward of the incoming gradient fused into the prologue
  W2S_CASE(16, 16, 3, 3, PRO_DNORM, EPI_ACT_BWD, false)
  W2S_CASE(32, 16, 3, 3, PRO_DNORM, EPI_ACT_BWD, false)
  W2S_CASE(32, 32, 3, 3, PRO_DNORM, EPI_ACT_BWD, false)
  W2S_CASE(64, 32, 3, 3, PRO_DNORM, EPI_ACT_BWD, false)
  W2S_CASE(64, 64, 3, 3, PRO_DNORM, EPI_ACT_BWD, false)
  W2S_CASE(128, 64, 3, 3, PRO_DNORM, EPI_ACT_BWD, false)
  W2S_CASE(128, 128, 3, 3, PRO_DNORM, EPI_ACT_BWD, false)
  W2S_CASE(16, 16, 1, 1, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(32, 16, 1, 1, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(32, 32, 1, 1, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(64, 32, 1, 1, PRO_NONE, EPI_PLAIN, false)
  W2S_CASE(64, 64, 1, 1, PRO_NONE, EPI_PLAIN, false)
#undef W2S_CASE
  return fail("conv1d: no kernel for cin=%d cout=%d taps=%d pro=%d epi=%d ds=%d", c.cin, c.cout, c.taps, c.prologue,
              c.epilogue, c.has_ds);
}

// Rotating slot allocator for inference workspaces.
struct Slots {
  uint8_t* base;
  size_t slot_bytes;
  int n;
  bool busy[8];
  void* get() {
    for (int i = 0; i < n; ++i)
      if (!busy[i]) {
        busy[i] = true;
        return base + (size_t)i * slot_bytes;
      }
    return nullptr;
  }
  void put(const void* p) {
    if (p == nullptr) return;
    const size_t i = ((const uint8_t*)p - base) / slot_bytes;
    if (i < (size_t)n) busy[i] = false;
  }
};

constexpr int kEncSlots = 5;

size_t enc_layer_stats_count(const w2s_encoder_desc* d, int B) {  // fp64 sum / sumsq accumulators of all conv layers
  size_t n = 0;
  for (int i = 0; i < d->n_blocks; ++i) n += (size_t)3 * B * d->channels[i] * 2;
  return n;
}
// + 4 doubles per sample for the raw-signal sums of the block-0 fusion (S0, R0, R1, R2)
size_t enc_stats_count(const w2s_encoder_desc* d, int B) { return enc_layer_stats_count(d, B) + (size_t)4 * B; }

int check_encoder_desc(const w2s_encoder_desc* d) {
  if (d == nullptr) return fail("encoder: null descriptor");
  if (d->n_blocks < 1 || d->n_blocks > W2S_MAX_BLOCKS) return fail("encoder: n_blocks=%d out of range", d->n_blocks);
  if (d->feature_dim != 128) return fail("encoder: feature_dim=%d (only 128 is built)", d->feature_dim);
  if (d->channels[0] != 16) return fail("encoder: initial_channels=%d (only 16 is built)", d->channels[0]);
  if (d->wide_blocks < 0 || d->wide_blocks >= d->n_blocks || (d->wide_blocks > 0 && d->channels[d->wide_blocks - 1] > 64))
    return fail("encoder: wide_blocks=%d must cover only leading blocks with <= 64 channels", d->wide_blocks);
  if (d->wide_blocks > 4 && (d->channels[4] != 64 || d->channels[3] != 32))
    return fail("encoder: wide_blocks=%d needs the 16,16,32,32,64,64 channel plan", d->wide_blocks);
  if (d->wide_blocks > 0 && (d->n_blocks < 2 || d->channels[1] != 16)) return fail("encoder: wide_blocks needs the fused block 0");
  if (d->wide_blocks & 1) return fail("encoder: wide_blocks=%d (only whole channel groups: 0, 2, 4 or 6 are built)", d->wide_blocks);
  return 0;
}

}  // namespace

extern "C" {

int w2s_abi_version(void) { return 11; }
const char* w2s_last_error(void) { return g_err.c_str(); }

int w2s_conv_uses_split(int cin, int cout) { return (cin <= 16 && cout <= 16) ? 1 : 0; }
int w2s_encoder_conv_split(int wide_blocks, int block, int cin, int cout) {
  if (w2s_conv_uses_split(cin, cout)) return 1;
  return (block < wide_blocks && cin <= 64 && cout <= 64) ? 1 : 0;  // every wide block carries split operands
}

size_t w2s_packed_conv_weight_bytes(int cout, int cin, int taps, int split) {
  return (size_t)cout * cin * taps * sizeof(__half) * (split ? 2 : 1);
}

int w2s_pack_conv_weight(const float* w, int cout, int cin, int taps, int taps_major, int split, void* out, void* stream) {
  if (w == nullptr || out == nullptr || cin % 8 != 0 || cout <= 0 || taps <= 0)
    return fail("pack_conv: bad arguments cin=%d cout=%d taps=%d", cin, cout, taps);
  const int total = cout * cin * taps;
  pack_conv_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, cout, cin, taps, taps_major, split, (__half*)out);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : cuda_fail(e, "pack_conv");
}

int w2s_pack_batch(const w2s_pack_job* jobs_device, int n_jobs, int max_elems, void* stream) {
  if (jobs_device == nullptr || n_jobs <= 0 || n_jobs > 65535 || max_elems <= 0) return fail("pack_batch: bad arguments");
  int gx = (max_elems + 255) / 256;
  if (gx > 64) gx = 64;  // grid-stride inside a job: keeps the launch at n_jobs x 64 blocks
  LaunchScope scope((cudaStream_t)stream, "pack_batch", 0, 0);
  pack_batch_kernel<<<dim3(gx, n_jobs), 256, 0, (cudaStream_t)stream>>>(jobs_device);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : cuda_fail(e, "pack_batch");
}

int w2s_pack_linear_frag(const float* w, int n, int k, void* out, void* stream) {
  if (w == nullptr || out == nullptr || n % 8 != 0 || k % 16 != 0) return fail("pack_frag: bad arguments n=%d k=%d", n, k);
  const int total = n * k;
  pack_frag_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, n, k, (__half*)out);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : cuda_fail(e, "pack_frag");
}

int w2s_stage_zscore(const void* raw, int raw_dtype, float* out, const uint8_t* present, double* ws, int B, int64_t T,
                     void* stream) {
  if (raw == nullptr || out == nullptr || ws == nullptr) return fail("stage_zscore: null pointer");
  if (B <= 0 || B > 65535 || T <= 0 || T % 4 != 0) return fail("stage_zscore: B=%d T=%lld (T must be a multiple of 4)", B, (long long)T);
  if (raw_dtype < 0 || raw_dtype > 2) return fail("stage_zscore: raw_dtype=%d (0 fp32, 1 fp16, 2 int16)", raw_dtype);
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(ws, 0, (size_t)B * 3 * sizeof(double), st);
  if (e != cudaSuccess) return cuda_fail(e, "stage_zscore memset");
  StageArgs a{raw, out, present, ws, (long long)T};
  long long gx = (T / 4 + 255) / 256;
  const long long cap = 8LL * sm_count() / B + 1;
  if (gx > cap) gx = cap;
  const dim3 grid((unsigned)gx, B);
  const double esz = raw_dtype == 0 ? 4.0 : 2.0;
  {
    LaunchScope scope(st, "stage_stats", (double)B * T * esz, 0);
    if (raw_dtype == 0) stage_stats_kernel<STAGE_F32><<<grid, 256, 0, st>>>(a);
    else if (raw_dtype == 1) stage_stats_kernel<STAGE_F16><<<grid, 256, 0, st>>>(a);
    else stage_stats_kernel<STAGE_I16><<<grid, 256, 0, st>>>(a);
  }
  {
    LaunchScope scope(st, "stage_apply", (double)B * T * (esz + 4.0), 0);
    if (raw_dtype == 0) stage_apply_kernel<STAGE_F32><<<grid, 256, 0, st>>>(a);
    else if (raw_dtype == 1) stage_apply_kernel<STAGE_F16><<<grid, 256, 0, st>>>(a);
    else stage_apply_kernel<STAGE_I16><<<grid, 256, 0, st>>>(a);
  }
  e = cudaGetLastError();
  return e == cudaSuccess ? 0 : cuda_fail(e, "stage_zscore launch");
}

int w2s_debug_timestamps(uint64_t* out16, uint64_t* cta1024) {
  if (out16 == nullptr) return fail("debug_timestamps: null pointer");
  cudaError_t e = cudaMemcpyFromSymbol(out16, g_stream_ts, 16 * sizeof(uint64_t));
  if (e == cudaSuccess && cta1024 != nullptr) e = cudaMemcpyFromSymbol(cta1024, g_stream_cta_ts, 1024 * sizeof(uint64_t));
  return e == cudaSuccess ? 0 : cuda_fail(e, "debug_timestamps");
}

int w2s_conv1d_fwd(const w2s_conv_call* call, void* stream) {
  if (call == nullptr) return fail("conv1d: null call");
  return conv_dispatch(*call, (cudaStream_t)stream);
}

int w2s_conv1d_fwd_pair(const w2s_conv_call* c0, const w2s_conv_call* c1, void* stream) {
  if (c0 == nullptr || c1 == nullptr) return fail("conv1d pair: null call");
  const int rc = conv_dispatch(*c0, (cudaStream_t)stream, c1);
  if (rc == kNotPaired)
    return fail("conv1d pair: no paired kernel for c%d->%d k%d s%d pro%d epi%d ds%d in_wide=%d out_wide=%d split=%d B=%d "
                "L_in=%d (or the two calls differ in shape or configuration)", c0->cin, c0->cout, c0->taps, c0->stride,
                c0->prologue, c0->epilogue, c0->has_ds, c0->in_wide, c0->out_wide, c0->force_split, c0->B, c0->L_in);
  return rc;
}

size_t w2s_encoder_workspace_bytes(const w2s_encoder_desc* d, int B, int64_t T, int keep) {
  if (check_encoder_desc(d) != 0 || B <= 0 || T <= 0) return 0;
  const size_t stats = align_up(enc_stats_count(d, B) * sizeof(double), 256);
  const size_t e = sizeof(__half);
  if (!keep) return stats + (size_t)kEncSlots * align_up((size_t)B * T * 16 * (d->wide_blocks > 0 ? 4 : e), 256);
  size_t act = 0;
  int64_t L = T;
  for (int i = 0; i < d->n_blocks; ++i) {
    const size_t c = d->channels[i];
    act += 2 * align_up((size_t)B * L * c * e, 256);        // y1, y2
    act += 2 * align_up((size_t)B * (L / 2) * c * e, 256);  // y3, r
    L /= 2;
  }
  return stats + act;
}

int w2s_encoder_layout(const w2s_encoder_desc* d, int B, int64_t T, int64_t* offsets) {
  // keep_activations = 1 layout: per block 7 byte offsets into the workspace: stats1, stats2, stats3, y1, r, y2, y3
  if (check_encoder_desc(d) != 0 || offsets == nullptr || B <= 0 || T <= 0) return fail("encoder_layout: bad arguments");
  const size_t stats_bytes = align_up(enc_stats_count(d, B) * sizeof(double), 256);
  size_t st = 0, act = stats_bytes;
  int64_t L = T;
  for (int i = 0; i < d->n_blocks; ++i) {
    const size_t c = d->channels[i], e = sizeof(__half);
    int64_t* o = offsets + 7 * i;
    for (int k = 0; k < 3; ++k) {
      o[k] = (int64_t)st;
      st += (size_t)B * c * 2 * sizeof(double);
    }
    o[3] = (int64_t)act; act += align_up((size_t)B * L * c * e, 256);        // y1
    o[4] = (int64_t)act; act += align_up((size_t)B * (L / 2) * c * e, 256);  // r
    o[5] = (int64_t)act; act += align_up((size_t)B * L * c * e, 256);        // y2
    o[6] = (int64_t)act; act += align_up((size_t)B * (L / 2) * c * e, 256);  // y3
    L /= 2;
  }
  return 0;
}

// One encoder forward as a list of launches: built first, then issued - singly (w2s_encoder_fwd) or zipped with the list of
// a second encoder of identical architecture, whose stream-kernel layers then share their launches (w2s_encoder_fwd_pair).
struct EncStep {
  enum Kind { MEMSET, XSTATS, FIRST, CONV } kind;
  w2s_conv_call cc;       // CONV
  void* ptr; size_t bytes;  // MEMSET
  XStatsArgs xa;          // XSTATS (+ the finalize kernel's arguments)
  const float* x; const double* xs; const float* w_first; const uint8_t* row_mask; double* s1;
  FirstConvArgs fa;       // FIRST
  int B, L;
};

static int encoder_plan(const w2s_encoder_desc* d, const float* x, int B, int64_t T, void* workspace, size_t ws_bytes,
                        int keep, void* z_out, uint8_t* row_mask, std::vector<EncStep>& plan) {
  if (check_encoder_desc(d) != 0) return 1;
  if (x == nullptr || z_out == nullptr || row_mask == nullptr || workspace == nullptr) return fail("encoder: null pointer");
  const int64_t spe = (int64_t)4 << d->n_blocks;  // samples per epoch = 2^(n_blocks+2)
  if (B <= 0 || T <= 0) return fail("encoder: empty input B=%d T=%lld", B, (long long)T);
  if (T % spe != 0) return fail("Input length %lld must be divisible by samples_per_epoch=%lld.", (long long)T, (long long)spe);
  if (T > 0x7fffffff / 2) return fail("encoder: T=%lld too long", (long long)T);
  const size_t need = w2s_encoder_workspace_bytes(d, B, T, keep);
  if (ws_bytes < need) return fail("encoder: workspace %zu < required %zu", ws_bytes, need);
  EncStep blank;
  memset(&blank, 0, sizeof(blank));
  auto emit_conv = [&](const w2s_conv_call& cc) {
    EncStep s = blank;
    s.kind = EncStep::CONV;
    s.cc = cc;
    plan.push_back(s);
  };

  const size_t stats_bytes = align_up(enc_stats_count(d, B) * sizeof(double), 256);
  double* stats = (double*)workspace;
  {
    EncStep s = blank;
    s.kind = EncStep::MEMSET;
    s.ptr = stats;
    s.bytes = stats_bytes;
    plan.push_back(s);
  }
  uint8_t* act_base = (uint8_t*)workspace + stats_bytes;

  Slots slots;
  memset(&slots, 0, sizeof(slots));
  slots.base = act_base;
  slots.slot_bytes = align_up((size_t)B * T * 16 * (!keep && d->wide_blocks > 0 ? 4 : sizeof(__half)), 256);
  auto wide = [&](int blk) { return !keep && blk >= 0 && blk < d->wide_blocks; };
  slots.n = kEncSlots;
  size_t bump = 0;
  auto alloc = [&](size_t bytes) -> void* {
    if (!keep) return slots.get();
    void* p = act_base + bump;
    bump += align_up(bytes, 256);
    return p;
  };
  auto release = [&](const void* p) {
    if (!keep) slots.put(p);
  };

  double* st_ptr = stats;
  auto next_stats = [&](int c) {
    double* p = st_ptr;
    st_ptr += (size_t)B * c * 2;
    return p;
  };

  int L = (int)T;
  const void* prev_y3 = nullptr;
  const void* prev_r = nullptr;
  const double* prev_s3 = nullptr;
  int prev_c = 1;
  for (int i = 0; i < d->n_blocks; ++i) {
    const int c = d->channels[i];
    const size_t e = sizeof(__half);
    void* y1 = alloc((size_t)B * L * c * e);
    void* r = alloc((size_t)B * (L / 2) * c * e);
    double* s1 = next_stats(c);
    double* s2 = next_stats(c);
    double* s3 = next_stats(c);
    if (y1 == nullptr || r == nullptr) return fail("encoder: slot allocator exhausted");
    const bool fuse0 = !keep && d->n_blocks >= 2 && d->channels[1] == 16;  // block-0 fusion (inference only)
    if (i == 0 && fuse0) {
      // conv1 of block 0 is recomputed inside conv2's prologue; only its statistics are needed up front
      release(y1);
      release(r);
      y1 = nullptr;
      r = nullptr;
      double* xs = stats + enc_layer_stats_count(d, B);  // zeroed with the rest of the statistics region
      XStatsArgs xa;
      xa.x = x; xa.xs = xs; xa.row_mask = row_mask; xa.T = L;
      EncStep s = blank;
      s.kind = EncStep::XSTATS;
      s.xa = xa; s.x = x; s.xs = xs; s.w_first = d->w_first; s.row_mask = row_mask; s.s1 = s1; s.B = B; s.L = L;
      plan.push_back(s);
    } else if (i == 0) {
      FirstConvArgs fa;
      fa.x = x;
      fa.w = d->w_first;
      fa.w_ds = d->w_first_ds;
      fa.y1 = (act_t*)y1;
      fa.r0 = (act_t*)r;
      fa.stats = s1;
      fa.row_mask = row_mask;
      fa.T = L;
      EncStep s = blank;
      s.kind = EncStep::FIRST;
      s.fa = fa; s.B = B; s.L = L;
      plan.push_back(s);
    } else {
      w2s_conv_call cc;
      memset(&cc, 0, sizeof(cc));
      cc.cin = prev_c; cc.cout = c; cc.taps = 3; cc.stride = 1; cc.dilation = 1; cc.pad = 1;
      cc.prologue = W2S_PRO_NORM_RES; cc.epilogue = W2S_EPI_STATS; cc.has_ds = 1;
      if (i == 1 && fuse0) {  // residual branch of block 0 recomputed from the raw signal
        cc.prologue = W2S_PRO_NORM_RES_X;
        cc.x_raw = x; cc.w_first_ds = d->w_first_ds; cc.T_raw = (int)T;
      }
      cc.B = B; cc.L_in = L; cc.L_out = L;
      cc.in = prev_y3; cc.in_res = prev_r; cc.in_stats = prev_s3;
      cc.w = d->w_conv[i][0]; cc.w_ds = d->w_ds[i];
      cc.out = y1; cc.out_ds = r; cc.out_stats = s1; cc.row_mask = row_mask; cc.in_eps = d->norm_eps;
      cc.in_wide = wide(i - 1); cc.out_wide = wide(i);
      cc.force_split = keep ? 0 : w2s_encoder_conv_split(d->wide_blocks, i, prev_c, c);
      emit_conv(cc);
      release(prev_y3);
      release(prev_r);
    }
    void* y2 = alloc((size_t)B * L * c * e);
    if (y2 == nullptr) return fail("encoder: slot allocator exhausted");
    {
      w2s_conv_call cc;
      memset(&cc, 0, sizeof(cc));
      cc.cin = c; cc.cout = c; cc.taps = 3; cc.stride = 1; cc.dilation = 1; cc.pad = 1;
      cc.prologue = W2S_PRO_NORM; cc.epilogue = W2S_EPI_STATS;
      if (i == 0 && fuse0) {
        cc.prologue = W2S_PRO_FIR;
        cc.x_raw = x; cc.w_first = d->w_first; cc.T_raw = (int)T;
      }
      cc.B = B; cc.L_in = L; cc.L_out = L;
      cc.in = y1; cc.in_stats = s1; cc.w = d->w_conv[i][1];
      cc.out = y2; cc.out_stats = s2; cc.row_mask = row_mask; cc.in_eps = d->norm_eps;
      cc.in_wide = wide(i) && !(i == 0 && fuse0); cc.out_wide = wide(i);
      cc.force_split = keep ? 0 : w2s_encoder_conv_split(d->wide_blocks, i, c, c);
      emit_conv(cc);
    }
    release(y1);
    void* y3 = alloc((size_t)B * (L / 2) * c * e);
    if (y3 == nullptr) return fail("encoder: slot allocator exhausted");
    {
      w2s_conv_call cc;
      memset(&cc, 0, sizeof(cc));
      cc.cin = c; cc.cout = c; cc.taps = 3; cc.stride = 2; cc.dilation = 1; cc.pad = 1;
      cc.prologue = W2S_PRO_NORM; cc.epilogue = W2S_EPI_STATS;
      cc.B = B; cc.L_in = L; cc.L_out = L / 2;
      cc.in = y2; cc.in_stats = s2; cc.w = d->w_conv[i][2];
      cc.out = y3; cc.out_stats = s3; cc.row_mask = row_mask; cc.in_eps = d->norm_eps;
      cc.in_wide = wide(i); cc.out_wide = wide(i);
      cc.force_split = keep ? 0 : w2s_encoder_conv_split(d->wide_blocks, i, c, c);
      emit_conv(cc);
    }
    release(y2);
    prev_y3 = y3;
    prev_r = r;
    prev_s3 = s3;
    prev_c = c;
    L /= 2;
  }
  {  // time-distributed Linear(4C -> F) + GELU  (models/wav2sleep.py:261-265)
    w2s_conv_call cc;
    memset(&cc, 0, sizeof(cc));
    cc.cin = prev_c; cc.cout = d->feature_dim; cc.taps = 4; cc.stride = 4; cc.dilation = 1; cc.pad = 0;
    cc.prologue = W2S_PRO_NORM_RES; cc.epilogue = W2S_EPI_BIAS_GELU;
    cc.B = B; cc.L_in = L; cc.L_out = L / 4;
    cc.in = prev_y3; cc.in_res = prev_r; cc.in_stats = prev_s3; cc.w = d->w_lin; cc.bias = d->b_lin;
    cc.out = z_out; cc.row_mask = row_mask; cc.in_eps = d->norm_eps;
    emit_conv(cc);
  }
  return 0;
}

// closed-form block-0 statistics of one signal, or of two signals of equal shape in the same two launches
static int run_x_stats(const EncStep& s, const EncStep* s2, cudaStream_t st) {
  const int n = s2 != nullptr ? 2 : 1;
  {
    LaunchScope scope(st, s2 != nullptr ? "x_stats x2" : "x_stats", n * (double)s.B * s.L * 4.0, n * (double)s.B * s.L * 8.0);
    int gx = (s.L / 4 + 255) / 256;
    const int cap = (4 * sm_count() + n * s.B - 1) / (n * s.B);  // ~4 long-lived blocks per SM over the whole batch
    if (gx > cap) gx = cap;
    const EncStep& t = s2 != nullptr ? *s2 : s;
    const XFinalizeArgs f0 = {s.x, s.xs, s.w_first, s.row_mask, s.s1}, f1 = {t.x, t.xs, t.w_first, t.row_mask, t.s1};
    x_stats_kernel<<<dim3(gx < 1 ? 1 : gx, s.B, n), 256, 0, st>>>(s.xa, t.xa);
    x_stats_finalize_kernel<<<dim3((s.B * 16 + 127) / 128, n), 128, 0, st>>>(f0, f1, s.B, s.L);
  }
  cudaError_t ce = cudaGetLastError();
  return ce == cudaSuccess ? 0 : cuda_fail(ce, "x_stats launch");
}

static int run_enc_step(const EncStep& s, cudaStream_t st) {
  switch (s.kind) {
    case EncStep::MEMSET: {
      cudaError_t ce = cudaMemsetAsync(s.ptr, 0, s.bytes, st);
      return ce == cudaSuccess ? 0 : cuda_fail(ce, "encoder memset");
    }
    case EncStep::XSTATS:
      return run_x_stats(s, nullptr, st);
    case EncStep::FIRST: {
      cudaError_t ce;
      {
        char fl_label[64];
        snprintf(fl_label, sizeof(fl_label), "first_conv c1->16 k3 B%d L%d", s.B, s.L);
        LaunchScope scope(st, fl_label, (double)s.B * s.L * (4.0 + 32.0 + 16.0), 2.0 * s.B * (double)s.L * 16 * 3.5);
        ce = launch_first_conv(s.fa, s.B, st);
      }
      return ce == cudaSuccess ? 0 : cuda_fail(ce, "first_conv launch");
    }
    case EncStep::CONV:
      return conv_dispatch(s.cc, st);
  }
  return fail("encoder: bad plan step");
}

int w2s_encoder_fwd(const w2s_encoder_desc* d, const float* x, int B, int64_t T, void* workspace, size_t ws_bytes,
                    int keep, void* z_out, uint8_t* row_mask, void* stream) {
  std::vector<EncStep> plan;
  if (encoder_plan(d, x, B, T, workspace, ws_bytes, keep, z_out, row_mask, plan) != 0) return 1;
  for (const EncStep& s : plan)
    if (run_enc_step(s, (cudaStream_t)stream) != 0) return 1;
  return 0;
}

int w2s_encoder_fwd_pair(const w2s_encoder_desc* d0, const float* x0, void* workspace0, void* z_out0, uint8_t* row_mask0,
                         const w2s_encoder_desc* d1, const float* x1, void* workspace1, void* z_out1, uint8_t* row_mask1,
                         int B, int64_t T, size_t ws_bytes, int keep, void* stream) {
  std::vector<EncStep> p0, p1;
  if (encoder_plan(d0, x0, B, T, workspace0, ws_bytes, keep, z_out0, row_mask0, p0) != 0) return 1;
  if (encoder_plan(d1, x1, B, T, workspace1, ws_bytes, keep, z_out1, row_mask1, p1) != 0) return 1;
  cudaStream_t st = (cudaStream_t)stream;
  bool same = p0.size() == p1.size();
  for (size_t i = 0; same && i < p0.size(); ++i) same = p0[i].kind == p1[i].kind;
  if (!same) {  // different architectures: one encoder after the other
    for (const EncStep& s : p0)
      if (run_enc_step(s, st) != 0) return 1;
    for (const EncStep& s : p1)
      if (run_enc_step(s, st) != 0) return 1;
    return 0;
  }
  for (size_t i = 0; i < p0.size(); ++i) {
    if (p0[i].kind == EncStep::CONV) {
      const int rc = conv_dispatch(p0[i].cc, st, &p1[i].cc);
      if (rc == 0) continue;
      if (rc != kNotPaired) return 1;
    }
    if (p0[i].kind == EncStep::XSTATS && p0[i].B == p1[i].B && p0[i].L == p1[i].L) {
      if (run_x_stats(p0[i], &p1[i], st) != 0) return 1;
      continue;
    }
    if (run_enc_step(p0[i], st) != 0 || run_enc_step(p1[i], st) != 0) return 1;
  }
  return 0;
}

int w2s_epoch_mixer_fwd(const w2s_mixer_desc* d, const void* const* z, const uint8_t* const* row_mask, int n_signals,
                        int B, int S, void* out, void* stream) {
  if (d == nullptr || z == nullptr || out == nullptr) return fail("epoch_mixer: null pointer");
  if (n_signals < 1) return fail("No signals provided to MultiModalAttentionEmbedder.");
  if (n_signals > W2S_MAX_SIGNALS) return fail("epoch_mixer: %d signals > %d", n_signals, W2S_MAX_SIGNALS);
  if (d->feature_dim != kMixF || d->n_heads != kMixHeads || d->dim_ff != kMixFF)
    return fail("epoch_mixer: only feature_dim=128, nhead=8, dim_ff=512 is built (got %d, %d, %d)", d->feature_dim,
                d->n_heads, d->dim_ff);
  if (d->n_layers < 1 || d->n_layers > W2S_MAX_MIXER_LAYERS) return fail("epoch_mixer: n_layers=%d", d->n_layers);
  if (B <= 0 || S <= 0) return fail("epoch_mixer: empty input");
  MixerArgs a;
  memset(&a, 0, sizeof(a));
  a.n_layers = d->n_layers;
  for (int l = 0; l < d->n_layers; ++l) {
    const w2s_mixer_layer& s = d->layer[l];
    MixerLayerW& w = a.layer[l];
    w.in_w = (const uint2*)s.in_w; w.out_w = (const uint2*)s.out_w;
    w.ff1_w = (const uint2*)s.ff1_w; w.ff2_w = (const uint2*)s.ff2_w;
    w.in_b = s.in_b; w.out_b = s.out_b; w.ff1_b = s.ff1_b; w.ff2_b = s.ff2_b;
    w.ln1_w = s.ln1_w; w.ln1_b = s.ln1_b; w.ln2_w = s.ln2_w; w.ln2_b = s.ln2_b;
  }
  for (int i = 0; i < n_signals; ++i) {
    if (z[i] == nullptr) return fail("epoch_mixer: z[%d] is null", i);
    a.z[i] = (const act_t*)z[i];
    a.row_mask[i] = row_mask ? row_mask[i] : nullptr;
  }
  a.cls = d->cls;
  a.out = (act_t*)out;
  a.n_epochs = B * S;
  a.S = S;
  a.ln_eps = d->ln_eps;
  cudaError_t e;
  {
    const double D = n_signals + 1;
    // layer flops (2*MAC): qkv 3F^2, out F^2, ffn 2*F*FF per token; last layer only K,V for all tokens + CLS row
    const double per_tok_full = 2.0 * (4.0 * 128 * 128 + 2.0 * 128 * 512);
    const double last = 2.0 * (D * 2.0 * 128 * 128 + 2.0 * 128 * 128 + 2.0 * 128 * 512);
    const double fl = (double)B * S * ((d->n_layers - 1) * D * per_tok_full + last);
    LaunchScope scope((cudaStream_t)stream, "epoch_mixer", (double)B * S * 128 * 2.0 * (n_signals + 1), fl);
    e = launch_epoch_mixer(a, n_signals, sm_count(), (cudaStream_t)stream);
  }
  return e == cudaSuccess ? 0 : cuda_fail(e, "epoch_mixer launch");
}

size_t w2s_seqmixer_workspace_bytes(const w2s_seq_desc* d, int B, int S, int keep) {
  if (d == nullptr || B <= 0 || S <= 0) return 0;
  const size_t t = align_up((size_t)B * S * 128 * sizeof(__half), 256);
  if (keep) return t * ((size_t)d->n_blocks * d->n_dilations + 1);
  const size_t fused = seq_fused_workspace_bytes(B, S, d->n_dilations);  // 0 when the shape is not served by it
  return t * 4 > fused ? t * 4 : fused;
}

int w2s_seqmixer_head_fwd(const w2s_seq_desc* d, const void* x, int B, int S, void* workspace, size_t ws_bytes,
                          int keep, void* feat_out, float* logits, void* stream) {
  if (d == nullptr || x == nullptr || workspace == nullptr || logits == nullptr) return fail("seqmixer: null pointer");
  if (d->feature_dim != 128 || d->kernel_size != 7) return fail("seqmixer: only feature_dim=128, kernel_size=7 is built");
  if (d->n_blocks < 1 || d->n_blocks > W2S_MAX_SEQ_BLOCKS || d->n_dilations < 1 || d->n_dilations > W2S_MAX_DILATIONS)
    return fail("seqmixer: n_blocks=%d n_dilations=%d", d->n_blocks, d->n_dilations);
  if (d->n_classes < 1 || d->n_classes > 8) return fail("seqmixer: n_classes=%d", d->n_classes);
  if (ws_bytes < w2s_seqmixer_workspace_bytes(d, B, S, keep)) return fail("seqmixer: workspace too small");
  const size_t t = align_up((size_t)B * S * 128 * sizeof(__half), 256);
  uint8_t* ws = (uint8_t*)workspace;
  SeqGeom geom;
  if (!keep && d->n_blocks * d->n_dilations <= kSeqMaxLayers && seq_fused_geometry(B, S, d->n_dilations, geom)) {
    // inference: all layers of a night inside one thread-block cluster (seq_mixer.cuh)
    SeqArgs a;
    memset(&a, 0, sizeof(a));
    for (int bl = 0; bl < d->n_blocks; ++bl)
      for (int k = 0; k < d->n_dilations; ++k) {
        const int l = bl * d->n_dilations + k;
        a.w[l] = (const act_t*)d->w[bl][k];
        a.ln_w[l] = d->ln_w[bl][k];
        a.ln_b[l] = d->ln_b[bl][k];
      }
    a.x = (const act_t*)x; a.buf = (act_t*)ws; a.feat_out = (act_t*)feat_out;
    a.head_w = d->head_w; a.head_b = d->head_b; a.logits = logits; a.n_classes = d->n_classes;
    a.n_blocks = d->n_blocks; a.n_dil = d->n_dilations; a.S = S; a.ln_eps = d->ln_eps;
    const double rows = (double)B * S, layers = (double)d->n_blocks * d->n_dilations;
    LaunchScope scope((cudaStream_t)stream, "seq_mixer fused", rows * 128 * 2.0 * 2.0 * layers,
                      2.0 * 7 * 128 * 128 * rows * layers);
    cudaError_t e = launch_seq_mixer(a, geom, B, (cudaStream_t)stream);
    return e == cudaSuccess ? 0 : cuda_fail(e, "seq_mixer launch");
  }
  // keep = 0: slots 0/1 ping-pong inside a block, slots 2/3 alternate as block outputs (a block's input is the
  // previous block's output or x, so it is never overwritten while it is still the residual source).
  int next = 0;
  const void* block_in = x;
  for (int bl = 0; bl < d->n_blocks; ++bl) {
    const void* cur = block_in;
    for (int k = 0; k < d->n_dilations; ++k) {
      const bool last_layer = (k == d->n_dilations - 1);
      const bool last_block = (bl == d->n_blocks - 1);
      void* o;
      if (last_layer && last_block && feat_out != nullptr) o = feat_out;
      else if (keep) o = ws + (size_t)(next++) * t;
      else o = ws + (size_t)(last_layer ? 2 + (bl & 1) : (k & 1)) * t;
      w2s_conv_call cc;
      memset(&cc, 0, sizeof(cc));
      cc.cin = 128; cc.cout = 128; cc.taps = 7; cc.stride = 1; cc.dilation = 1 << k; cc.pad = 3 << k;
      cc.prologue = W2S_PRO_NONE;
      cc.epilogue = last_layer ? W2S_EPI_LN_GELU_RES : W2S_EPI_LN_GELU;
      cc.B = B; cc.L_in = S; cc.L_out = S;
      cc.in = cur; cc.w = d->w[bl][k]; cc.ln_w = d->ln_w[bl][k]; cc.ln_b = d->ln_b[bl][k];
      cc.out = o; cc.ln_eps = d->ln_eps;
      if (last_layer) cc.res = block_in;
      if (last_layer && last_block) {
        cc.head_w = d->head_w; cc.head_b = d->head_b; cc.logits = logits; cc.n_classes = d->n_classes;
      }
      if (conv_dispatch(cc, (cudaStream_t)stream) != 0) return 1;
      cur = o;
    }
    block_in = cur;
  }
  return 0;
}

// ================================================================================================
// training path: kernel-level entry points (orchestrated by wav2sleep_b200/training.py)
// ================================================================================================
#define W2S_LAUNCH_CHECK(what)                                       \
  do {                                                               \
    cudaError_t e__ = cudaGetLastError();                            \
    if (e__ != cudaSuccess) return cuda_fail(e__, what);             \
    return 0;                                                        \
  } while (0)

static int ew_grid(long long work_items, int threads = 256) {
  long long g = (work_items + threads - 1) / threads;
  const long long cap = 8LL * sm_count();
  if (g > cap) g = cap;
  return g < 1 ? 1 : (int)g;
}

int w2s_gemm_tn(const void* X, const void* Y, float* Cm, int M, int N, int taps, int tap_stride, int B, int LX, int LY,
                int y_stride, int y_offset, long long ldc_m, long long ldc_n, long long ldc_t, float scale,
                const uint8_t* row_mask, void* stream) {
  if (!X || !Y || !Cm || B <= 0 || LX <= 0 || LY <= 0 || y_stride < 1 || taps < 1 || taps > 16) return fail("gemm_tn: bad arguments");
  // taps == 3 with unit tap stride on narrow operands: fused kernel (X and Y read once); else one grid slice per tap
  const bool fused = (taps == 3 && tap_stride == 1 && y_stride == 1 && M <= 64 && N <= 64);
  GemmTNArgs a;
  a.X = (const act_t*)X; a.Y = (const act_t*)Y; a.C = Cm; a.row_mask = row_mask;
  a.B = B; a.LX = LX; a.LY = LY; a.y_stride = y_stride; a.y_offset = y_offset;
  a.ldc_m = ldc_m; a.ldc_n = ldc_n; a.ldc_t = ldc_t; a.scale = scale;
  a.grid_taps = fused ? 1 : taps; a.tap_stride = tap_stride;
  cudaStream_t st = (cudaStream_t)stream;
  char label[64];
  snprintf(label, sizeof(label), "gemm_tn %dx%d t%d B%d L%d", M, N, taps, B, LX);
  const int ktaps = fused ? 3 : 1;
  LaunchScope scope(st, label, (double)B * LX * (M + N) * 2.0, 2.0 * B * (double)LX * M * N * taps);
  cudaError_t e = cudaErrorInvalidValue;
#define W2S_TN(MM, NN, TT) if (M == MM && N == NN && ktaps == TT) e = launch_gemm_tn<MM, NN, TT>(a, sm_count(), st);
  W2S_TN(16, 16, 1) W2S_TN(32, 16, 1) W2S_TN(32, 32, 1) W2S_TN(64, 32, 1) W2S_TN(64, 64, 1) W2S_TN(128, 64, 1)
  W2S_TN(128, 128, 1) W2S_TN(16, 16, 3) W2S_TN(32, 16, 3) W2S_TN(32, 32, 3) W2S_TN(64, 32, 3) W2S_TN(64, 64, 3)
#undef W2S_TN
  if (e == cudaErrorInvalidValue) return fail("gemm_tn: no kernel for M=%d N=%d taps=%d", M, N, taps);
  return e == cudaSuccess ? 0 : cuda_fail(e, "gemm_tn launch");
}

// The encoder element kernels keep one 8-channel chunk per thread for the whole grid-stride loop (C / 8 a power of two
// dividing 256) and their per-channel constants in 128-entry shared-memory slots.
static bool enc_channels_ok(int Cc) { return Cc == 8 || Cc == 16 || Cc == 32 || Cc == 64 || Cc == 128; }

int w2s_enc_act_fwd(const void* y, const void* r, const double* stats, void* a, const uint8_t* row_mask, int B, int L,
                    int Cc, float eps, void* stream) {
  if (!y || !stats || !a) return fail("enc_act_fwd: bad arguments");
  if (!enc_channels_ok(Cc)) return fail("enc_act_fwd: C=%d (built for 8, 16, 32, 64 or 128 channels)", Cc);
  EncActArgs p{(const act_t*)y, (const act_t*)r, stats, (act_t*)a, row_mask, B, L, Cc, eps};
  LaunchScope scope((cudaStream_t)stream, "enc_act_fwd", (double)B * L * Cc * (r ? 6.0 : 4.0), 0);
  dim3 grid(ew_grid((long long)L * (Cc / 8)), B);
  enc_act_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("enc_act_fwd");
}

int w2s_enc_act_bwd(const void* dout, const void* y, const void* r, const double* stats, void* dxh, void* dr, double* sums,
                    void* a_out, const uint8_t* row_mask, int B, int L, int Cc, float eps, void* stream) {
  if (!dout || !y || !stats || !dxh || !sums) return fail("enc_act_bwd: bad arguments");
  if (!enc_channels_ok(Cc)) return fail("enc_act_bwd: C=%d (built for 8, 16, 32, 64 or 128 channels)", Cc);
  if (r && !dr) return fail("enc_act_bwd: dr missing");
  EncActBwdArgs p{(const act_t*)dout, (const act_t*)y, (const act_t*)r, stats, (act_t*)dxh, (act_t*)dr, sums, row_mask,
                  B, L, Cc, eps, (act_t*)a_out};
  LaunchScope scope((cudaStream_t)stream, "enc_act_bwd", (double)B * L * Cc * ((r ? 10.0 : 6.0) + (a_out ? 2.0 : 0.0)), 0);
  const int rows_per_block = 256 / (Cc / 8);
  int gx = (L + rows_per_block * 8 - 1) / (rows_per_block * 8);
  if (gx > 4 * sm_count()) gx = 4 * sm_count();
  dim3 grid(gx < 1 ? 1 : gx, B);
  enc_act_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("enc_act_bwd");
}

int w2s_enc_norm_bwd(const void* dxh, const void* y, const double* stats, const double* sums, void* dy,
                     const uint8_t* row_mask, int B, int L, int Cc, int upsample, float eps, void* stream) {
  if (!dxh || !y || !stats || !sums || !dy) return fail("enc_norm_bwd: bad arguments");
  if (!enc_channels_ok(Cc)) return fail("enc_norm_bwd: C=%d (built for 8, 16, 32, 64 or 128 channels)", Cc);
  EncNormBwdArgs p{(const act_t*)dxh, (const act_t*)y, stats, sums, (act_t*)dy, row_mask, B, L, Cc, upsample, eps};
  LaunchScope scope((cudaStream_t)stream, "enc_norm_bwd", (double)B * L * Cc * 6.0, 0);
  dim3 grid(ew_grid((long long)L * (Cc / 8)), B);
  enc_norm_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("enc_norm_bwd");
}

int w2s_first_conv_wgrad(const float* x, const void* dy1, const void* dr, float* dw1, float* dwds, const uint8_t* row_mask,
                         int B, int T, float scale, void* stream) {
  if (!x || !dy1 || !dr || !dw1 || !dwds) return fail("first_conv_wgrad: bad arguments");
  // dr holds the T / 2 rows of the stride-2 residual branch: row l / 2 pairs with input sample l for even l
  if (B <= 0 || T <= 0 || (T & 1)) return fail("first_conv_wgrad: B=%d T=%d (needs B > 0 and an even T > 0)", B, T);
  FirstWgradArgs p{x, (const act_t*)dy1, (const act_t*)dr, dw1, dwds, row_mask, B, T, scale};
  LaunchScope scope((cudaStream_t)stream, "first_conv_wgrad", (double)B * T * (4.0 + 32.0 + 16.0), 0);
  int gx = (T + 256 * 16 - 1) / (256 * 16);
  dim3 grid(gx < 1 ? 1 : gx, B);
  first_conv_wgrad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("first_conv_wgrad");
}

int w2s_first_conv_dgrad(const float* x, const void* dy1, const void* dr, const float* w1, const float* wds,
                         const uint8_t* row_mask, float* dx, int B, int T, float scale, void* stream) {
  if (!x || !dy1 || !dr || !w1 || !wds || !row_mask || !dx)
    return fail("first_conv_dgrad: NULL operand (x=%p dy1=%p dr=%p w1=%p wds=%p row_mask=%p dx=%p)", (const void*)x, dy1, dr,
                (const void*)w1, (const void*)wds, (const void*)row_mask, (void*)dx);
  if (B <= 0 || B > 65535 || T <= 0 || (T & 1))
    return fail("first_conv_dgrad: B=%d T=%d (needs 0 < B <= 65535 and an even T > 0)", B, T);
  FirstDgradArgs p{x, (const act_t*)dy1, (const act_t*)dr, w1, wds, row_mask, dx, (long long)T, scale};
  LaunchScope scope((cudaStream_t)stream, "first_conv_dgrad", (double)B * T * (32.0 + 16.0 + 4.0 + 4.0), (double)B * T * 128.0);
  dim3 grid((unsigned)(((long long)T + kFirstDgradThreads - 1) / kFirstDgradThreads), B);
  first_conv_dgrad_kernel<<<grid, kFirstDgradThreads, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("first_conv_dgrad");
}

int w2s_row_ln_fwd(const void* x, const void* res, const float* g, const float* b, void* out, long long rows, int gelu,
                   float eps, void* stream) {
  if (!x || !g || !b || !out || rows <= 0) return fail("row_ln_fwd: bad arguments");
  RowLnArgs p;
  memset(&p, 0, sizeof(p));
  p.x = (const act_t*)x; p.res = (const act_t*)res; p.g = g; p.b = b; p.out = (act_t*)out; p.rows = rows; p.gelu = gelu;
  p.eps = eps;
  LaunchScope scope((cudaStream_t)stream, "row_ln_fwd", (double)rows * 128 * (res ? 6.0 : 4.0), 0);
  row_ln_fwd_kernel<<<ew_grid(rows * 32), 256, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("row_ln_fwd");
}

int w2s_row_ln_bwd(const void* x, const void* res, const float* g, const float* b, const void* dout, const void* dadd,
                   void* dx, void* ds, float* dg, float* db, long long rows, int gelu, float eps, float gscale,
                   void* stream) {
  if (!x || !g || !b || !dout || !dx || !dg != !db || rows <= 0) return fail("row_ln_bwd: bad arguments");
  RowLnArgs p;
  memset(&p, 0, sizeof(p));
  p.x = (const act_t*)x; p.res = (const act_t*)res; p.g = g; p.b = b; p.out = (act_t*)dx; p.dout = (const act_t*)dout;
  p.dadd = (const act_t*)dadd; p.ds = (act_t*)ds; p.dg = dg; p.db = db; p.rows = rows; p.gelu = gelu; p.eps = eps;
  p.gscale = gscale;
  LaunchScope scope((cudaStream_t)stream, "row_ln_bwd", (double)rows * 128 * 8.0, 0);
  int gx = ew_grid(rows * 32);
  if (gx > 2 * sm_count()) gx = 2 * sm_count();
  row_ln_bwd_kernel<<<gx, 256, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("row_ln_bwd");
}

int w2s_gelu_fwd(const void* pre, void* out, long long n, void* stream) {
  if (!pre || !out || n <= 0 || n % 8) return fail("gelu_fwd: bad arguments");
  LaunchScope scope((cudaStream_t)stream, "gelu_fwd", (double)n * 4.0, 0);
  gelu_fwd_kernel<<<ew_grid(n / 8), 256, 0, (cudaStream_t)stream>>>((const act_t*)pre, (act_t*)out, n / 8);
  W2S_LAUNCH_CHECK("gelu_fwd");
}
int w2s_gelu_bwd(const void* pre, const void* dout, void* din, long long n, void* stream) {
  if (!pre || !dout || !din || n <= 0 || n % 8) return fail("gelu_bwd: bad arguments");
  LaunchScope scope((cudaStream_t)stream, "gelu_bwd", (double)n * 6.0, 0);
  gelu_bwd_kernel<<<ew_grid(n / 8), 256, 0, (cudaStream_t)stream>>>((const act_t*)pre, (const act_t*)dout, (act_t*)din, n / 8);
  W2S_LAUNCH_CHECK("gelu_bwd");
}

int w2s_colsum(const void* x, float* out, long long rows, int Cc, int row_stride, int row_offset, const uint8_t* row_mask,
               long long rows_per_sample, float scale, void* stream) {
  if (!x || !out || rows <= 0 || Cc % 8 || Cc > 128 || 256 % (Cc / 8)) return fail("colsum: bad arguments");
  LaunchScope scope((cudaStream_t)stream, "colsum", (double)rows * Cc * 2.0, 0);
  int gx = ew_grid(rows * (Cc / 8));
  if (gx > 2 * sm_count()) gx = 2 * sm_count();
  colsum_kernel<<<gx, 256, 0, (cudaStream_t)stream>>>((const act_t*)x, out, rows, Cc, row_stride > 0 ? row_stride : 1,
                                                      row_offset, row_mask, rows_per_sample > 0 ? rows_per_sample : rows,
                                                      scale);
  W2S_LAUNCH_CHECK("colsum");
}

int w2s_attn_fwd(const void* q, const void* k, const void* v, void* o, const uint8_t* key_mask, int N, int D, float drop_p,
                 uint64_t seed, uint32_t site, void* stream) {
  if (!q || !k || !v || !o || N <= 0 || D < 1 || D > 5) return fail("attn_fwd: bad arguments");
  if (!(drop_p >= 0.0f && drop_p < 1.0f)) return fail("attn_fwd: dropout p=%g outside [0, 1)", drop_p);
  AttnArgs p;
  memset(&p, 0, sizeof(p));
  p.drop_p = drop_p; p.seed = seed; p.site = site;
  p.q = (const act_t*)q; p.k = (const act_t*)k; p.v = (const act_t*)v; p.o = (act_t*)o; p.key_mask = key_mask; p.N = N; p.D = D;
  LaunchScope scope((cudaStream_t)stream, "attn_fwd", (double)N * D * 128 * 8.0, 0);
  attn_kernel<false><<<(N * 8 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("attn_fwd");
}
int w2s_attn_bwd(const void* q, const void* k, const void* v, const void* dout, void* dq, void* dk, void* dv,
                 const uint8_t* key_mask, int N, int D, float drop_p, uint64_t seed, uint32_t site, void* stream) {
  if (!q || !k || !v || !dout || !dq || !dk || !dv || N <= 0 || D < 1 || D > 5) return fail("attn_bwd: bad arguments");
  if (!(drop_p >= 0.0f && drop_p < 1.0f)) return fail("attn_bwd: dropout p=%g outside [0, 1)", drop_p);
  AttnArgs p;
  memset(&p, 0, sizeof(p));
  p.drop_p = drop_p; p.seed = seed; p.site = site;
  p.q = (const act_t*)q; p.k = (const act_t*)k; p.v = (const act_t*)v; p.dout = (const act_t*)dout;
  p.dq = (act_t*)dq; p.dk = (act_t*)dk; p.dv = (act_t*)dv; p.key_mask = key_mask; p.N = N; p.D = D;
  LaunchScope scope((cudaStream_t)stream, "attn_bwd", (double)N * D * 128 * 14.0, 0);
  attn_kernel<true><<<(N * 8 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("attn_bwd");
}

int w2s_dropout(const void* x, const void* res, void* out, uint8_t* mask_out, int64_t n, float p, uint64_t seed, uint32_t site,
                void* stream) {
  if (n <= 0 || n % 8 != 0 || n > 0xffffffffLL) return fail("dropout: n=%lld must be a positive multiple of 8", (long long)n);
  if (!(p >= 0.0f && p < 1.0f)) return fail("dropout: p=%g outside [0, 1)", p);
  if (mask_out == nullptr && (x == nullptr || out == nullptr)) return fail("dropout: null pointer");
  DropArgs a;
  a.x = (const act_t*)x; a.res = (const act_t*)res; a.out = (act_t*)out; a.mask_out = mask_out;
  a.n = n; a.p = p; a.seed = seed; a.site = site;
  LaunchScope scope((cudaStream_t)stream, "dropout", (double)n * (res ? 6.0 : 4.0), 0);
  dropout_kernel<<<(unsigned)((n / 8 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
  W2S_LAUNCH_CHECK("dropout");
}

int w2s_tokens_fwd(const void* const* z, const uint8_t* const* row_mask, const float* cls, void* tokens, uint8_t* key_mask,
                   int N, int S, int n_sig, void* stream) {
  if (!z || !cls || !tokens || !key_mask || n_sig < 1 || n_sig > 4) return fail("tokens_fwd: bad arguments");
  TokenArgs p;
  memset(&p, 0, sizeof(p));
  for (int i = 0; i < n_sig; ++i) { p.z[i] = (const act_t*)z[i]; p.row_mask[i] = row_mask ? row_mask[i] : nullptr; }
  p.cls = cls; p.tokens = (act_t*)tokens; p.key_mask = key_mask; p.N = N; p.S = S; p.n_sig = n_sig;
  LaunchScope scope((cudaStream_t)stream, "tokens_fwd", (double)N * (n_sig + 1) * 128 * 4.0, 0);
  tokens_fwd_kernel<<<ew_grid((long long)N * (n_sig + 1) * 16), 256, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("tokens_fwd");
}
int w2s_tokens_bwd(const void* dtokens, void* const* dz, const uint8_t* const* row_mask, float* dcls, int N, int S, int n_sig,
                   float cls_scale, void* stream) {
  if (!dtokens || !dz || n_sig < 1 || n_sig > 4) return fail("tokens_bwd: bad arguments");
  TokenArgs p;
  memset(&p, 0, sizeof(p));
  for (int i = 0; i < n_sig; ++i) { p.dz[i] = (act_t*)dz[i]; p.row_mask[i] = row_mask ? row_mask[i] : nullptr; }
  p.dtokens = (const act_t*)dtokens; p.dcls = dcls; p.N = N; p.S = S; p.n_sig = n_sig; p.cls_scale = cls_scale;
  LaunchScope scope((cudaStream_t)stream, "tokens_bwd", (double)N * (n_sig + 1) * 128 * 4.0, 0);
  int gx = ew_grid((long long)N * (n_sig + 1) * 16);
  if (gx > 2 * sm_count()) gx = 2 * sm_count();
  tokens_bwd_kernel<<<gx, 256, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("tokens_bwd");
}
int w2s_rows_gather(const void* in, void* out, long long n_rows, int stride, int offset, int scatter, void* stream) {
  if (!in || !out || n_rows <= 0 || stride < 1) return fail("rows_gather: bad arguments");
  LaunchScope scope((cudaStream_t)stream, "rows_gather", (double)n_rows * 128 * 4.0, 0);
  rows_gather_kernel<<<ew_grid(n_rows * 16), 256, 0, (cudaStream_t)stream>>>((const act_t*)in, (act_t*)out, n_rows, stride,
                                                                          offset, scatter);
  W2S_LAUNCH_CHECK("rows_gather");
}

int w2s_head_fwd(const void* feat, const float* w, const float* b, float* logits, long long N, int Cc, void* stream) {
  if (!feat || !w || !b || !logits || N <= 0 || Cc < 1 || Cc > 8) return fail("head_fwd: bad arguments");
  HeadArgs p;
  memset(&p, 0, sizeof(p));
  p.feat = (const act_t*)feat; p.w = w; p.b = b; p.logits = logits; p.N = N; p.C = Cc;
  LaunchScope scope((cudaStream_t)stream, "head_fwd", (double)N * 128 * 2.0, 0);
  head_fwd_kernel<<<ew_grid(N * 32), 256, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("head_fwd");
}
int w2s_ce_fwd_bwd(const float* logits, const long long* labels, long long N, int Cc, long long ignore_index, double* scratch2,
                   float* loss, float* dlogits, void* stream) {
  if (!logits || !labels || !scratch2 || !loss || !dlogits || N <= 0 || Cc < 1 || Cc > 8) return fail("ce_fwd_bwd: bad arguments");
  HeadArgs p;
  memset(&p, 0, sizeof(p));
  p.logits = (float*)logits; p.labels = labels; p.loss_sum = scratch2; p.count = scratch2 + 1; p.loss = loss; p.N = N; p.C = Cc;
  p.ignore_index = ignore_index;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(scratch2, 0, 2 * sizeof(double), st);
  if (e != cudaSuccess) return cuda_fail(e, "ce memset");
  LaunchScope scope(st, "ce_fwd_bwd", (double)N * Cc * 8.0, 0);
  ce_loss_kernel<<<ew_grid(N), 256, 0, st>>>(p);
  ce_grad_kernel<<<ew_grid(N), 256, 0, st>>>(p, dlogits);
  W2S_LAUNCH_CHECK("ce_fwd_bwd");
}
int w2s_head_bwd(const void* feat, const float* w, const float* dlogits, void* dfeat, float* dw, float* db, long long N, int Cc,
                 float dfeat_scale, void* stream) {
  if (!feat || !w || !dlogits || !dfeat || N <= 0 || Cc < 1 || Cc > 8) return fail("head_bwd: bad arguments");
  HeadArgs p;
  memset(&p, 0, sizeof(p));
  p.feat = (const act_t*)feat; p.w = w; p.dlogits = dlogits; p.dfeat = (act_t*)dfeat; p.dw = dw; p.db = db; p.N = N; p.C = Cc;
  p.dfeat_scale = dfeat_scale;
  LaunchScope scope((cudaStream_t)stream, "head_bwd", (double)N * 128 * 4.0, 0);
  int gx = ew_grid(N * 32);
  if (gx > sm_count()) gx = sm_count();
  head_bwd_kernel<<<gx, 256, 0, (cudaStream_t)stream>>>(p);
  W2S_LAUNCH_CHECK("head_bwd");
}

int w2s_sumsq(const float* g, long long n, double* out, void* stream) {
  if (!g || !out || n <= 0) return fail("sumsq: bad arguments");
  LaunchScope scope((cudaStream_t)stream, "sumsq", (double)n * 4.0, 0);
  int gx = ew_grid(n);
  if (gx > 2 * sm_count()) gx = 2 * sm_count();
  sumsq_kernel<<<gx, 256, 0, (cudaStream_t)stream>>>(g, n, out);
  W2S_LAUNCH_CHECK("sumsq");
}
int w2s_absmax(const float* g, long long n, float* out, void* stream) {
  if (!g || !out || n <= 0) return fail("absmax: bad arguments (g=%p out=%p n=%lld)", (const void*)g, (void*)out, n);
  cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float), (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "absmax memset");
  LaunchScope scope((cudaStream_t)stream, "absmax", (double)n * 4.0, 0);
  int gx = ew_grid(n);
  if (gx > 2 * sm_count()) gx = 2 * sm_count();
  absmax_kernel<<<gx, 256, 0, (cudaStream_t)stream>>>(g, n, reinterpret_cast<unsigned int*>(out));
  W2S_LAUNCH_CHECK("absmax");
}
int w2s_ig_path_inputs(const float* x, const float* x0, const float* alphas, int K, int B, int T, float* out,
                       void* stream) {
  if (!x || !alphas || !out)
    return fail("ig_path_inputs: NULL operand (x=%p alphas=%p out=%p)", (const void*)x, (const void*)alphas, (void*)out);
  if (K < 1 || B < 1 || T < 1) return fail("ig_path_inputs: K=%d B=%d T=%d (each must be >= 1)", K, B, T);
  const long long n = (long long)B * T;
  LaunchScope scope((cudaStream_t)stream, "ig_path_inputs", (double)n * (x0 ? 8.0 : 4.0) + (double)n * K * 4.0, (double)n * K * 2.0);
  ig::path_inputs_kernel<<<ew_grid(n, ig::kThreads), ig::kThreads, 0, (cudaStream_t)stream>>>(x, x0, alphas, K, n, out);
  W2S_LAUNCH_CHECK("ig_path_inputs");
}
int w2s_ig_accumulate(const float* grads, const float* weights, int K, const float* x, const float* x0, int B, int T,
                      float* attr, int first, void* stream) {
  if (!grads || !weights || !x || !attr)
    return fail("ig_accumulate: NULL operand (grads=%p weights=%p x=%p attr=%p)", (const void*)grads, (const void*)weights,
                (const void*)x, (void*)attr);
  if (K < 1 || B < 1 || T < 1 || (first != 0 && first != 1))
    return fail("ig_accumulate: K=%d B=%d T=%d first=%d (K, B, T >= 1, first 0 or 1)", K, B, T, first);
  const long long n = (long long)B * T;
  LaunchScope scope((cudaStream_t)stream, "ig_accumulate", (double)n * (4.0 * K + (x0 ? 8.0 : 4.0) + (first ? 4.0 : 8.0)),
                    (double)n * (2.0 * K + 1.0));
  ig::accumulate_kernel<<<ew_grid(n, ig::kThreads), ig::kThreads, 0, (cudaStream_t)stream>>>(grads, weights, K, x, x0, n, attr,
                                                                                           first);
  W2S_LAUNCH_CHECK("ig_accumulate");
}
int w2s_adamw_step(float* p_, const float* g, float* m, float* v, long long n, const double* gnorm_sq, float lr, float beta1,
                   float beta2, float eps, float weight_decay, float max_norm, float grad_scale, long long step, float* ema,
                   float ema_decay, void* stream) {
  if (!p_ || !g || !m || !v || n <= 0 || step < 1) return fail("adamw_step: bad arguments");
  if (ema != nullptr && !(ema_decay >= 0.0f && ema_decay <= 1.0f)) return fail("decay must be in [0, 1], got %g", ema_decay);
  AdamWArgs a;
  a.p = p_; a.g = g; a.m = m; a.v = v; a.n = n; a.gnorm_sq = gnorm_sq; a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps;
  a.weight_decay = weight_decay; a.max_norm = max_norm; a.grad_scale = grad_scale;
  a.bias_c1 = (float)(1.0 - pow((double)beta1, (double)step));
  a.bias_c2 = (float)(1.0 - pow((double)beta2, (double)step));
  a.ema = ema; a.ema_decay = ema_decay;
  LaunchScope scope((cudaStream_t)stream, "adamw_step", (double)n * (ema ? 36.0 : 28.0), (double)n * 12.0);
  adamw_kernel<<<ew_grid(n), 256, 0, (cudaStream_t)stream>>>(a);
  W2S_LAUNCH_CHECK("adamw_step");
}

// ================================================================================================
// general fp32 path for non-default model options (general.cuh), orchestrated by wav2sleep_b200/general.py
// ================================================================================================
int w2s_gen_conv(const float* in, const float* w, const float* bias, float* out, const uint8_t* row_mask, int B, int L_in,
                 int L_out, int cin, int cout, int taps, int stride, int dil, int pad_left, int taps_major,
                 int raw_inf_to_zero, void* stream) {
  if (!in || !w || !out || B <= 0 || B > 65535 || L_in <= 0 || L_out <= 0 || cin < 1 || cout < 1 || taps < 1 || stride < 1 || dil < 1)
    return fail("gen_conv: bad arguments (B=%d L_in=%d L_out=%d cin=%d cout=%d taps=%d)", B, L_in, L_out, cin, cout, taps);
  gen::ConvArgs a{in, w, bias, out, row_mask, B, L_in, L_out, cin, cout, taps, stride, dil, pad_left, taps_major, raw_inf_to_zero};
  long long gx = ((long long)L_out * cout + 255) / 256;
  const long long cap = 32LL * sm_count() / B + 1;
  if (gx > cap) gx = cap;
  LaunchScope scope((cudaStream_t)stream, "gen_conv", 0, 2.0 * B * (double)L_out * cout * cin * taps);
  gen::conv_kernel<<<dim3((unsigned)gx, B), 256, 0, (cudaStream_t)stream>>>(a);
  W2S_LAUNCH_CHECK("gen_conv");
}
int w2s_gen_stats(const float* x, double* stats, const uint8_t* row_mask, int B, int L, int Cc, void* stream) {
  if (!x || !stats || B <= 0 || B > 65535 || L <= 0 || Cc < 1) return fail("gen_stats: bad arguments");
  LaunchScope scope((cudaStream_t)stream, "gen_stats", (double)B * L * Cc * 4.0, 0);
  gen::stats_kernel<<<dim3(Cc, B), 256, 0, (cudaStream_t)stream>>>(x, stats, row_mask, L, Cc);
  W2S_LAUNCH_CHECK("gen_stats");
}
int w2s_gen_norm_consts(const double* stats, const float* weight, const float* bias, const float* running_mean,
                        const float* running_var, float* scale, float* shift, int B, int Cc, int L, int mode, int groups,
                        float eps, void* stream) {
  if (!scale || !shift || B <= 0 || Cc < 1 || mode < 0 || mode > 2) return fail("gen_norm_consts: bad arguments");
  if (mode == gen::NORM_BATCH_EVAL ? (!running_mean || !running_var) : !stats) return fail("gen_norm_consts: statistics missing");
  if (mode == gen::NORM_GROUP && (groups < 1 || Cc % groups)) return fail("gen_norm_consts: %d channels, %d groups", Cc, groups);
  gen::NormConstArgs a{stats, weight, bias, running_mean, running_var, scale, shift, B, Cc, L, mode, groups, eps};
  LaunchScope scope((cudaStream_t)stream, "gen_norm_consts", 0, 0);
  gen::norm_consts_kernel<<<ew_grid((long long)B * Cc), 256, 0, (cudaStream_t)stream>>>(a);
  W2S_LAUNCH_CHECK("gen_norm_consts");
}
int w2s_gen_affine_act(const float* in, const float* scale, const float* shift, const float* res, float* out,
                       const uint8_t* row_mask, int B, int L, int Cc, int act, int per_channel, void* stream) {
  if (!in || !out || B <= 0 || B > 65535 || L <= 0 || Cc < 1 || act < 0 || act > 4) return fail("gen_affine_act: bad arguments");
  gen::AffineActArgs a{in, scale, shift, res, out, row_mask, B, L, Cc, act, per_channel};
  long long gx = ((long long)L * Cc + 255) / 256;
  const long long cap = 32LL * sm_count() / B + 1;
  if (gx > cap) gx = cap;
  LaunchScope scope((cudaStream_t)stream, "gen_affine_act", (double)B * L * Cc * 8.0, 0);
  gen::affine_act_kernel<<<dim3((unsigned)gx, B), 256, 0, (cudaStream_t)stream>>>(a);
  W2S_LAUNCH_CHECK("gen_affine_act");
}
int w2s_gen_rownorm(const float* x, const float* weight, const float* bias, float* out, long long rows, int Cc, int rms, int act,
                    float eps, void* stream) {
  if (!x || !out || rows <= 0 || Cc < 1 || act < 0 || act > 4) return fail("gen_rownorm: bad arguments");
  gen::RowNormArgs a{x, weight, bias, out, rows, Cc, rms, act, eps};
  LaunchScope scope((cudaStream_t)stream, "gen_rownorm", (double)rows * Cc * 8.0, 0);
  gen::rownorm_kernel<<<ew_grid(rows * 32), 256, 0, (cudaStream_t)stream>>>(a);
  W2S_LAUNCH_CHECK("gen_rownorm");
}
int w2s_gen_attn(const float* q, const float* k, const float* v, float* o, const uint8_t* key_mask, int N, int D, int H, int hd,
                 int ld, float drop_p, uint64_t seed, uint32_t site, void* stream) {
  if (!q || !k || !v || !o || N <= 0 || D < 1 || H < 1 || hd < 1 || ld < H * hd) return fail("gen_attn: bad arguments");
  if (!(drop_p >= 0.0f && drop_p < 1.0f)) return fail("gen_attn: dropout p=%g outside [0, 1)", drop_p);
  gen::AttnArgs a{q, k, v, o, key_mask, N, D, H, hd, ld, drop_p, seed, site};
  LaunchScope scope((cudaStream_t)stream, "gen_attn", (double)N * D * H * hd * 16.0, 0);
  gen::attn_kernel<<<ew_grid((long long)N * D * H, 128), 128, 0, (cudaStream_t)stream>>>(a);
  W2S_LAUNCH_CHECK("gen_attn");
}

// ---- backward of the general path ----
static bool gen_conv_shape_ok(int B, int L_in, int L_out, int cin, int cout, int taps, int stride, int dil) {
  return B > 0 && B <= 65535 && L_in > 0 && L_out > 0 && cin >= 1 && cout >= 1 && taps >= 1 && stride >= 1 && dil >= 1;
}
int w2s_gen_conv_dgrad(const float* dout, const float* w, float* din, const uint8_t* row_mask, int B, int L_in, int L_out, int cin,
                       int cout, int taps, int stride, int dil, int pad_left, int taps_major, void* stream) {
  if (!dout || !w || !din || !gen_conv_shape_ok(B, L_in, L_out, cin, cout, taps, stride, dil))
    return fail("gen_conv_dgrad: bad arguments (B=%d L_in=%d L_out=%d cin=%d cout=%d taps=%d)", B, L_in, L_out, cin, cout, taps);
  gen::ConvBwdArgs a{nullptr, w, dout, din, nullptr, row_mask, B, L_in, L_out, cin, cout, taps, stride, dil, pad_left,
                     taps_major, 0};
  long long gx = ((long long)L_in * cin + 255) / 256;
  const long long cap = 32LL * sm_count() / B + 1;
  if (gx > cap) gx = cap;
  LaunchScope scope((cudaStream_t)stream, "gen_conv_dgrad", 4.0 * B * ((double)L_out * cout + (double)L_in * cin),
                    2.0 * B * (double)L_out * cout * cin * taps);
  gen::conv_dgrad_kernel<<<dim3((unsigned)gx, B), 256, 0, (cudaStream_t)stream>>>(a);
  W2S_LAUNCH_CHECK("gen_conv_dgrad");
}
int w2s_gen_conv_wgrad(const float* in, const float* dout, float* dw, float* dbias, double* ws, const uint8_t* row_mask, int B,
                       int L_in, int L_out, int cin, int cout, int taps, int stride, int dil, int pad_left, int taps_major,
                       int raw_inf_to_zero, void* stream) {
  if (!in || !dout || !ws || (!dw && !dbias) || !gen_conv_shape_ok(B, L_in, L_out, cin, cout, taps, stride, dil))
    return fail("gen_conv_wgrad: bad arguments (B=%d L_in=%d L_out=%d cin=%d cout=%d taps=%d)", B, L_in, L_out, cin, cout, taps);
  const long long K = (long long)taps * cin * cout;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(ws, 0, (size_t)(K + cout) * sizeof(double), st);
  if (e != cudaSuccess) return cuda_fail(e, "gen_conv_wgrad memset");
  gen::ConvBwdArgs a{in, nullptr, dout, nullptr, ws, row_mask, B, L_in, L_out, cin, cout, taps, stride, dil, pad_left, taps_major,
                     raw_inf_to_zero};
  const long long gx = (K + 31) / 32, tiles = ((long long)B * L_out + gen::kRedTile - 1) / gen::kRedTile;
  // enough position tiles to fill the GPU ~8 blocks deep, each block walking several tiles (fewer fp64 atomics)
  long long gy = (8LL * sm_count() + gx - 1) / gx;
  if (gy > tiles) gy = tiles;
  if (gy > 65535) gy = 65535;
  if (gy < 1) gy = 1;
  LaunchScope scope(st, "gen_conv_wgrad", 4.0 * B * ((double)L_out * cout + (double)L_in * cin),
                    2.0 * B * (double)L_out * cout * cin * taps);
  gen::conv_wgrad_kernel<<<dim3((unsigned)gx, (unsigned)gy), 256, 0, st>>>(a);
  gen::conv_wgrad_finalize_kernel<<<ew_grid(K + cout), 256, 0, st>>>(a, dw, dbias);
  W2S_LAUNCH_CHECK("gen_conv_wgrad");
}
int w2s_gen_affine_act_bwd(const float* in, const float* scale, const float* shift, const float* res, const float* dout, float* din,
                           float* dpre, double* sums, const uint8_t* row_mask, int B, int L, int Cc, int act, int per_channel,
                           void* stream) {
  if (!in || !dout || B <= 0 || B > 65535 || L <= 0 || Cc < 1 || act < 0 || act > 4) return fail("gen_affine_act_bwd: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (sums) {
    cudaError_t e = cudaMemsetAsync(sums, 0, (size_t)(per_channel ? 1 : B) * Cc * 2 * sizeof(double), st);
    if (e != cudaSuccess) return cuda_fail(e, "gen_affine_act_bwd memset");
  }
  gen::AffineActBwdArgs a{in, scale, shift, res, dout, din, dpre, sums, row_mask, B, L, Cc, act, per_channel};
  const long long gx = (Cc + 31) / 32, tiles = ((long long)L + gen::kRedTile - 1) / gen::kRedTile;
  long long gy = (8LL * sm_count() + gx * B - 1) / (gx * B);
  if (gy > tiles) gy = tiles;
  if (gy > 65535) gy = 65535;
  if (gy < 1) gy = 1;
  LaunchScope scope(st, "gen_affine_act_bwd", (double)B * L * Cc * (4.0 * (2 + (res != nullptr) + (din != nullptr) + (dpre != nullptr))), 0);
  gen::affine_act_bwd_kernel<<<dim3((unsigned)gx, (unsigned)gy, B), 256, 0, st>>>(a);
  W2S_LAUNCH_CHECK("gen_affine_act_bwd");
}
int w2s_gen_norm_bwd(const float* x, const float* dpre, const double* stats, const double* sums, const float* weight, float* coef,
                     float* dx, float* dweight, float* dbias, const uint8_t* row_mask, int B, int L, int Cc, int groups, float eps,
                     void* stream) {
  if (!x || !dpre || !stats || !sums || !coef || !dx || B <= 0 || B > 65535 || L <= 0 || Cc < 1 || groups < 1 || Cc % groups)
    return fail("gen_norm_bwd: bad arguments (B=%d L=%d C=%d groups=%d)", B, L, Cc, groups);
  cudaStream_t st = (cudaStream_t)stream;
  gen::NormBwdArgs a{stats, sums, weight, row_mask, coef, dweight, dbias, B, Cc, L, groups, eps};
  LaunchScope scope(st, "gen_norm_bwd", (double)B * L * Cc * 12.0, 0);
  gen::norm_bwd_coef_kernel<<<ew_grid(Cc), 256, 0, st>>>(a);
  long long gx = ((long long)L * Cc + 255) / 256;
  const long long cap = 32LL * sm_count() / B + 1;
  if (gx > cap) gx = cap;
  gen::norm_bwd_apply_kernel<<<dim3((unsigned)gx, B), 256, 0, st>>>(x, dpre, coef, dx, row_mask, L, Cc);
  W2S_LAUNCH_CHECK("gen_norm_bwd");
}
int w2s_gen_rownorm_bwd(const float* x, const float* weight, const float* bias, const float* dout, float* dx, float* dweight,
                        float* dbias, double* ws, long long rows, int Cc, int rms, int act, float eps, void* stream) {
  if (!x || !dout || !dx || rows <= 0 || Cc < 1 || Cc > 2048 || act < 0 || act > 4 || ((dweight || dbias) && !ws))
    return fail("gen_rownorm_bwd: bad arguments (rows=%lld C=%d)", rows, Cc);
  cudaStream_t st = (cudaStream_t)stream;
  if (ws) {
    cudaError_t e = cudaMemsetAsync(ws, 0, (size_t)2 * Cc * sizeof(double), st);
    if (e != cudaSuccess) return cuda_fail(e, "gen_rownorm_bwd memset");
  }
  gen::RowNormBwdArgs a{x, weight, bias, dout, dx, ws, rows, Cc, rms, act, eps};
  int gx = ew_grid(rows * 32);
  if (gx > 2 * sm_count()) gx = 2 * sm_count();  // every block adds its 2 * C column partials once
  LaunchScope scope(st, "gen_rownorm_bwd", (double)rows * Cc * 12.0, 0);
  gen::rownorm_bwd_kernel<<<gx, 256, 2 * Cc * sizeof(double), st>>>(a);
  if (ws) gen::rownorm_bwd_finalize_kernel<<<ew_grid(Cc), 256, 0, st>>>(ws, dweight, dbias, Cc);
  W2S_LAUNCH_CHECK("gen_rownorm_bwd");
}
int w2s_gen_attn_bwd(const float* q, const float* k, const float* v, const float* dout, float* dq, float* dk, float* dv,
                     const uint8_t* key_mask, int N, int D, int H, int hd, int ld, float drop_p, uint64_t seed, uint32_t site,
                     void* stream) {
  if (!q || !k || !v || !dout || !dq || !dk || !dv || N <= 0 || D < 1 || H < 1 || hd < 1 || ld < H * hd)
    return fail("gen_attn_bwd: bad arguments");
  if (!(drop_p >= 0.0f && drop_p < 1.0f)) return fail("gen_attn_bwd: dropout p=%g outside [0, 1)", drop_p);
  gen::AttnBwdArgs a{q, k, v, dout, dq, dk, dv, key_mask, N, D, H, hd, ld, drop_p, seed, site};
  LaunchScope scope((cudaStream_t)stream, "gen_attn_bwd", (double)N * D * H * hd * 28.0, 0);
  gen::attn_bwd_kernel<<<ew_grid((long long)N * D * H, 128), 128, 0, (cudaStream_t)stream>>>(a);
  W2S_LAUNCH_CHECK("gen_attn_bwd");
}
int w2s_gen_bn_eval_bwd(const float* dscale, const float* dshift, const float* running_mean, const float* running_var,
                        float* dweight, float* dbias, int Cc, float eps, void* stream) {
  if (!dscale || !dshift || !running_mean || !running_var || (!dweight && !dbias) || Cc < 1)
    return fail("gen_bn_eval_bwd: bad arguments (C=%d)", Cc);
  LaunchScope scope((cudaStream_t)stream, "gen_bn_eval_bwd", (double)Cc * 24.0, 0);
  gen::bn_eval_bwd_kernel<<<ew_grid(Cc), 256, 0, (cudaStream_t)stream>>>(dscale, dshift, running_mean, running_var, dweight,
                                                                          dbias, Cc, eps);
  W2S_LAUNCH_CHECK("gen_bn_eval_bwd");
}
int w2s_gen_bn_stats(const float* x, double* stats, long long rows, int Cc, void* stream) {
  if (!x || !stats || rows < 1 || Cc < 1) return fail("gen_bn_stats: bad arguments (rows=%lld C=%d)", rows, Cc);
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(stats, 0, (size_t)Cc * 2 * sizeof(double), st);
  if (e != cudaSuccess) return cuda_fail(e, "gen_bn_stats memset");
  // blocks: enough row steps to keep 8 blocks on every SM, never more than there are steps
  const int cw = Cc < gen::kBnThreads ? Cc : gen::kBnThreads;
  const long long step = (long long)(gen::kBnThreads / cw) * gen::kBnUnroll;
  long long g = (rows + step - 1) / step;
  if (g > 8LL * sm_count()) g = 8LL * sm_count();
  LaunchScope scope(st, "gen_bn_stats", (double)rows * Cc * 4.0, (double)rows * Cc * 3.0);
  gen::bn_stats_kernel<<<(unsigned)g, gen::kBnThreads, 0, st>>>(x, stats, rows, Cc);
  gen::bn_stats_finalize_kernel<<<ew_grid(Cc), 256, 0, st>>>(x, stats, rows, Cc);
  W2S_LAUNCH_CHECK("gen_bn_stats");
}
int w2s_gen_bn_update_running(const double* stats, long long n, float* running_mean, float* running_var,
                              long long* num_batches_tracked, double momentum, int Cc, void* stream) {
  if (!stats || !running_mean || !running_var || !num_batches_tracked || Cc < 1)
    return fail("gen_bn_update_running: bad arguments (C=%d)", Cc);
  if (n < 2) return fail("gen_bn_update_running: Expected more than 1 value per channel when training, got n=%lld", n);
  LaunchScope scope((cudaStream_t)stream, "gen_bn_running", (double)Cc * 32.0 + 16.0, 0);
  gen::bn_update_running_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(stats, n, running_mean, running_var,
                                                                      num_batches_tracked, momentum, Cc);
  W2S_LAUNCH_CHECK("gen_bn_update_running");
}
int w2s_gen_dropout(const float* x, float* out, uint8_t* mask_out, long long n, float p, uint64_t seed, uint32_t site,
                    void* stream) {
  if (n <= 0 || n > 0xffffffffLL) return fail("gen_dropout: n=%lld outside [1, 2^32)", n);
  if (!(p >= 0.0f && p < 1.0f)) return fail("gen_dropout: p=%g outside [0, 1)", p);
  if (mask_out == nullptr && (x == nullptr || out == nullptr)) return fail("gen_dropout: null pointer");
  LaunchScope scope((cudaStream_t)stream, "gen_dropout", (double)n * (mask_out ? 1.0 : 8.0), 0);
  gen::dropout_kernel<<<ew_grid(n), 256, 0, (cudaStream_t)stream>>>(x, out, mask_out, n, p, seed, site);
  W2S_LAUNCH_CHECK("gen_dropout");
}

int w2s_gen_seq_stream_step(const w2s_gen_seq_stream_desc* d, const float* x_new, float* logits, int N, int R, long long pos,
                            void* stream) {
  if (!d || !x_new || !logits || N <= 0 || R <= 0 || pos < 0)
    return fail("gen_seq_stream_step: bad arguments (N=%d R=%d pos=%lld)", N, R, pos);
  const int F = d->feature_dim, k = d->kernel_size, nb = d->n_blocks, nd = d->n_dilations;
  if (F < 1 || F > W2S_STREAM_MAX_FEATURES)
    return fail("gen_seq_stream_step: feature_dim %d outside [1, W2S_STREAM_MAX_FEATURES = %d]", F, W2S_STREAM_MAX_FEATURES);
  if (k < 1 || k > W2S_STREAM_MAX_KERNEL)
    return fail("gen_seq_stream_step: kernel_size %d outside [1, W2S_STREAM_MAX_KERNEL = %d]", k, W2S_STREAM_MAX_KERNEL);
  if (nd < 1 || nd > W2S_STREAM_MAX_DILATIONS)
    return fail("gen_seq_stream_step: n_dilations %d outside [1, W2S_STREAM_MAX_DILATIONS = %d]", nd, W2S_STREAM_MAX_DILATIONS);
  if (nb < 1 || nb * nd > W2S_STREAM_MAX_LAYERS)
    return fail("gen_seq_stream_step: n_blocks %d x n_dilations %d outside [1, W2S_STREAM_MAX_LAYERS = %d]", nb, nd,
                W2S_STREAM_MAX_LAYERS);
  if (d->n_classes < 1 || !d->head_w) return fail("gen_seq_stream_step: classifier missing (n_classes=%d)", d->n_classes);
  if (d->norm < W2S_SEQ_NORM_NONE || d->norm > W2S_SEQ_NORM_RMS || d->act < 0 || d->act > 4)
    return fail("gen_seq_stream_step: norm %d / act %d unknown", d->norm, d->act);
  if (k > 1 && !d->ring) return fail("gen_seq_stream_step: ring state missing");
  for (int l = 0; l < nb * nd; ++l) {
    const w2s_gen_seq_stream_layer& L = d->layer[l];
    if (!L.w || (d->norm == W2S_SEQ_NORM_BATCH && (!L.running_mean || !L.running_var)))
      return fail("gen_seq_stream_step: parameters of layer %d missing", l);
  }
  // a tile of G * spt streams per CTA: enough CTAs to spread small N over the SMs, at most kStreamMaxAcc per thread
  const int G = gen::kStreamThreads / F, ld = F | 1;
  int cc = 8192 / (k * ld);
  cc = cc < 1 ? 1 : (cc > F ? F : cc);
  int spt = (int)(((long long)N + (long long)G * sm_count() - 1) / ((long long)G * sm_count()));
  spt = spt < 1 ? 1 : (spt > gen::kStreamMaxAcc ? gen::kStreamMaxAcc : spt);
  // shared memory fits at every spt: TS * F <= 8 * 256, so tile rows take <= 2048 * (k + 2) floats, and the weight chunk
  // cc * k * (F | 1) <= 8192 floats: <= 176 KB for k <= 16
  const size_t smem = gen::seq_stream_smem_floats(F, k, G * spt, cc) * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(gen::seq_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "gen_seq_stream_step smem attribute");
  gen::SeqStreamArgs a{*d, x_new, logits, N, R, pos, G, spt, cc};
  const int TS = G * spt;
  const long long grid = ((long long)N + TS - 1) / TS;
  const double ring_bytes = 4.0 * N * R * nb * (double)k * nd * F;  // k - 1 tap rows read + 1 row written per layer
  LaunchScope scope((cudaStream_t)stream, "gen_seq_stream_step", ring_bytes + 4.0 * N * R * (F + d->n_classes),
                    2.0 * N * R * (double)nb * nd * F * F * k);
  gen::seq_stream_kernel<<<(unsigned)grid, gen::kStreamThreads, smem, (cudaStream_t)stream>>>(a);
  W2S_LAUNCH_CHECK("gen_seq_stream_step");
}

int w2s_set_conv_impl(int impl) {
  if (impl != 0 && impl != 1 && impl != 3) return fail("set_conv_impl: %d", impl);
  g_conv_impl.store(impl);
  return 0;
}

long long w2s_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int w2s_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (auto& r : g_prof) {
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
  }
  g_prof.clear();
  g_prof_on = on != 0;
  return 0;
}

int w2s_profile_count(void) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  return (int)g_prof.size();
}

int w2s_profile_get(int i, char* label, int label_cap, float* ms, double* bytes, double* flops) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (i < 0 || i >= (int)g_prof.size() || label == nullptr || ms == nullptr) return fail("profile_get: bad index %d", i);
  const ProfRec& r = g_prof[i];
  cudaError_t e = cudaEventSynchronize(r.e1);
  if (e != cudaSuccess) return cuda_fail(e, "profile_get sync");
  e = cudaEventElapsedTime(ms, r.e0, r.e1);
  if (e != cudaSuccess) return cuda_fail(e, "profile_get elapsed");
  snprintf(label, label_cap, "%s", r.label.c_str());
  if (bytes) *bytes = r.bytes;
  if (flops) *flops = r.flops;
  return 0;
}

int w2s_argmax(const float* logits, int64_t n, int n_classes, int64_t* out, void* stream) {
  if (logits == nullptr || out == nullptr || n <= 0 || n_classes <= 0) return fail("argmax: bad arguments");
  const int grid = (int)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096);
  LaunchScope scope((cudaStream_t)stream, "argmax", (double)n * (n_classes * 4.0 + 8.0), 0.0);
  argmax_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(logits, (long long)n, n_classes, (long long*)out);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : cuda_fail(e, "argmax");
}

}  // extern "C"
