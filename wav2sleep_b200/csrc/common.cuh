// Shared device helpers for the wav2sleep B200 kernels (sm_100a only).
//
// Everything here is a thin inline-PTX wrapper: mbarrier, proxy fences, tcgen05
// (TMEM alloc / MMA / commit / ld), UMMA descriptors for the no-swizzle K-major
// canonical layout, fp16 packing and the fast GELU used in conv prologues.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace w2s {

// Storage/operand element type of every activation tensor and MMA operand.
// fp16 (not bf16): measured with the reference model, bf16 storage of the encoder
// activations gives 7.6e-2 max-abs logit error / 98.6 % argmax agreement, fp16 gives
// 1.0e-2 / 99.9 % (DESIGN.md "Numerics").  fp32 accumulation everywhere.
typedef __half act_t;

#define W2S_DEVINL __device__ __forceinline__

W2S_DEVINL uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
W2S_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
W2S_DEVINL void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
W2S_DEVINL bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// try_wait with a suspend-time hint: the hardware may park the warp for up to `ns` nanoseconds (it is woken when the
// phase completes), so a waiting role does not burn issue slots.  ncu on the round-1 kernels: 25 % of all executed
// warp instructions were the spin loops of waiting roles (try_wait + clock64 + compare + branch), taken from the same
// schedulers the transform warps issue on.
W2S_DEVINL bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}
// Bounded wait: a lost arrive turns into a trap (launch error) instead of a hung GPU.  The bound is an iteration count
// (no clock reads in the loop): 2^22 parked waits of up to 20 us each.
W2S_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t it = 0;
  while (!mbar_try_wait_hint(bar, parity, 20000u)) {
    if (++it > (1u << 22)) __trap();
  }
}

// One lane of a fully converged warp (warp-uniform code keeps operands in uniform registers, so single-thread
// instructions such as tcgen05.mma / cp.async.bulk need no per-lane waterfall loop).
W2S_DEVINL bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, px;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// 256-bit global store (STG.256, sm_100+): one instruction per 32-byte row chunk halves the LSU wavefronts of the
// row-per-lane epilogue stores.  Address must be 32-byte aligned.
W2S_DEVINL void stg256(void* ptr, const uint32_t (&v)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(ptr), "r"(v[0]), "r"(v[1]), "r"(v[2]),
               "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

// 16 consecutive fp16 channels of one row (32-byte aligned) in one store
W2S_DEVINL void store_h16(__half* dst, const float (&v)[16]);

// ----------------------------------------------------------------------------------------------
// fences
// ----------------------------------------------------------------------------------------------
// generic-proxy smem writes -> visible to the async proxy (tcgen05.mma operand reads)
W2S_DEVINL void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
W2S_DEVINL void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
W2S_DEVINL void tc_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// TMEM
// ----------------------------------------------------------------------------------------------
// Whole warp must call.  ncols: power of two in [32, 512].
W2S_DEVINL void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
W2S_DEVINL void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 covers fp16 and bf16 operands, fp32 accum.
W2S_DEVINL void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives (count 1) on the mbarrier once every previously issued tcgen05.mma of this thread is done.
W2S_DEVINL void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// 32 lanes x 16 consecutive fp32 columns: thread i of warp w reads TMEM lane 32*(w%4)+i.
W2S_DEVINL void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// 32 lanes x 32 / 64 consecutive fp32 columns in one instruction (one tcgen05.wait::ld per 32 / 64 columns instead of
// one per 16: the load round trip, not the instruction count, is what an epilogue warp waits for)
W2S_DEVINL void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
W2S_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// UMMA descriptors (cute/arch/mma_sm100_desc.hpp bit layout; SWIZZLE_NONE, K-major)
// ----------------------------------------------------------------------------------------------
// Canonical no-swizzle K-major operand: core matrix = 8 rows x 16 bytes, rows 16 B apart.
//   LBO = byte distance between the two 16-byte K chunks of one K=16 step
//   SBO = byte distance between consecutive 8-row groups along M/N
// With "chunk-major" staging [chunk][row][16 B] the rows of one chunk are contiguous, so SBO = 128 and
// a start address may be shifted by any number of rows (16 B each): that is how conv taps are addressed.
W2S_DEVINL uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (sm_100)
  return d;                // base_offset 0, lbo_mode 0, layout_type 0 (SWIZZLE_NONE)
}
// The same descriptor in two 32-bit halves.  Within one staged operand only the start-address field (low 14 bits, units
// of 16 bytes) changes from MMA to MMA, and it cannot carry into the LBO field because shared-memory addresses stay
// below 256 KB: a descriptor is `umma_desc(lo0 + (byte_offset >> 4), hi)` - ONE integer add on the issuing thread
// instead of shift / mask / or per operand (the MMA issuer of the 16-channel kernels was 95 % busy on this arithmetic).
W2S_DEVINL uint32_t umma_desc_lo(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
__host__ __device__ constexpr uint32_t umma_desc_hi(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14); }
W2S_DEVINL uint64_t umma_desc(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }
// kind::f16 instruction descriptor: fp32 accumulate, A/B both K-major, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N, bool bf16) {
  return (1u << 4)                      // c_format = F32
         | ((bf16 ? 1u : 0u) << 7)      // a_format
         | ((bf16 ? 1u : 0u) << 10)     // b_format
         | ((uint32_t)(N >> 3) << 17)   // n_dim
         | ((uint32_t)(M >> 4) << 24);  // m_dim
}

// ----------------------------------------------------------------------------------------------
// math
// ----------------------------------------------------------------------------------------------
// GELU(x) = x * Phi(x) with Phi(x) ~= 1 / (1 + exp(-2 xc (a + b xc^2 + c xc^4))), xc = clamp(x, +-5).
// Fitted against the erf form (reference models/utils.py:67-68 -> nn.GELU()): max abs error 2.5e-5 over R,
// 10x below fp16 rounding of the result.  One ex2 + one rcp on the MUFU pipe.
W2S_DEVINL float gelu_fast(float x) {
  const float xc = fminf(fmaxf(x, -5.0f), 5.0f);
  const float t = xc * xc;
  // coefficients pre-multiplied by -2*log2(e)
  float q = fmaf(t, 1.01448193e-3f, -0.10677673f);
  q = fmaf(q, t, -2.30112048f);
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(xc * q));
  return __fdividef(x, 1.0f + e);
}
// Two elements at once on the packed-fp32 pipe (FFMA2/FMUL2/FADD2, sm_100): ~half the issue slots of gelu_fast.
// 0.5 x (1 + tanh(x p(min(x^2,25)))) with ONE MUFU.TANH per element (tanh.approx.f32, 2^-11 relative error: below
// fp16 rounding of the result).  Clamping t = x^2 (not x) keeps the argument monotone for |x| > 5: u = x * p(25),
// |u| >= 7.5, tanh saturates.  Measured against a packed ex2+rcp form of gelu_fast: same logit parity (cardio 9e-3 /
// 100 %, EOG 2.2e-2 / 99.7 %), 10 % faster step.
W2S_DEVINL float2 gelu_fast2(float2 x) {
  float2 t = __fmul2_rn(x, x);
  t.x = fminf(t.x, 25.0f);
  t.y = fminf(t.y, 25.0f);
  float2 q = __ffma2_rn(t, make_float2(-3.5159264e-4f, -3.5159264e-4f), make_float2(0.037005995f, 0.037005995f));
  q = __ffma2_rn(q, t, make_float2(0.79750759f, 0.79750759f));
  const float2 u = __fmul2_rn(x, q);
  float2 th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th.x) : "f"(u.x));
  asm("tanh.approx.f32 %0, %1;" : "=f"(th.y) : "f"(u.y));
  const float2 h = __fmul2_rn(x, make_float2(0.5f, 0.5f));
  return __ffma2_rn(h, th, h);
}
W2S_DEVINL uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
// Compacted list of the samples a row mask leaves alive (mask[b] == 0), built by ONE WARP: all loads of the mask are
// issued before the first ballot (one global-memory round trip instead of one per sample on a single thread - the
// serial scan cost every launch ~2 us of set-up).  Returns the number of live samples.
W2S_DEVINL int build_live_list(const uint8_t* __restrict__ mask, int n, uint16_t* live, int lane) {
  int count = 0;
#pragma unroll 1
  for (int r0 = 0; r0 < n; r0 += 128) {
    uint8_t m[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int b = r0 + j * 32 + lane;
      m[j] = b < n ? mask[b] : (uint8_t)1;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const bool alive = m[j] == 0;
      const unsigned bal = __ballot_sync(0xffffffffu, alive);
      if (alive) live[count + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)(r0 + j * 32 + lane);
      count += __popc(bal);
    }
  }
  return count;
}
// 16 bytes of a tensor written by an earlier launch, streamed past L1
W2S_DEVINL uint4 ldg128_stream(const void* ptr) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(ptr));
  return v;
}
W2S_DEVINL void sts128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// Exact-erf GELU for low-volume epilogues.
W2S_DEVINL float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }

// {lo, hi} -> packed fp16x2, round-to-nearest, saturating to +-65504 instead of inf.
W2S_DEVINL uint32_t pack_h2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
// {lo, hi} -> packed bf16x2, round-to-nearest (bf16 operand measurement hook)
W2S_DEVINL uint32_t pack_bf2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
W2S_DEVINL float2 unpack_h2(uint32_t u) {
  __half2 h = *reinterpret_cast<__half2*>(&u);
  return __half22float2(h);
}

W2S_DEVINL void store_h16(__half* dst, const float (&v)[16]) {
  const uint32_t w[8] = {pack_h2(v[0], v[1]),   pack_h2(v[2], v[3]),   pack_h2(v[4], v[5]),   pack_h2(v[6], v[7]),
                         pack_h2(v[8], v[9]),   pack_h2(v[10], v[11]), pack_h2(v[12], v[13]), pack_h2(v[14], v[15])};
  stg256(dst, w);
}

// Transposing butterfly reduction over the 32 lanes of a warp for 16 per-lane values.
// On return lane l holds in v[0] the full 32-lane sum of channel ((l >> 1) & 15).
W2S_DEVINL int butterfly16_channel(int lane) { return (lane >> 1) & 15; }
W2S_DEVINL void butterfly16(float* v, int lane) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const bool hi = lane & 16;
    float send = hi ? v[i] : v[i + 8];
    float keep = hi ? v[i + 8] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool hi = lane & 8;
    float send = hi ? v[i] : v[i + 4];
    float keep = hi ? v[i + 4] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const bool hi = lane & 4;
    float send = hi ? v[i] : v[i + 2];
    float keep = hi ? v[i + 2] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  {
    const bool hi = lane & 2;
    float send = hi ? v[0] : v[1];
    float keep = hi ? v[1] : v[0];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
}

// ----------------------------------------------------------------------------------------------
// training-path element math shared by train_kernels.cuh and the fused dgrad epilogue of conv_igemm.cuh
// ----------------------------------------------------------------------------------------------
// tanh-form GELU and derivative (same fitted exponent as the forward prologue, one MUFU.TANH): used on the whole-night
// encoder tensors where erff/expf would make the element-wise kernels compute bound.
W2S_DEVINL float gelu_tanh(float x) {
  const float t = fminf(x * x, 25.0f);
  const float q = fmaf(fmaf(t, -3.5159264e-4f, 0.037005995f), t, 0.79750759f);
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(x * q));
  const float h = 0.5f * x;
  return fmaf(h, th, h);
}
W2S_DEVINL float gelu_grad_tanh(float x) {
  const float x2 = x * x;
  const float t = fminf(x2, 25.0f);
  const float q = fmaf(fmaf(t, -3.5159264e-4f, 0.037005995f), t, 0.79750759f);
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(x * q));
  const float dq = x2 < 25.0f ? 2.0f * x2 * fmaf(t, -7.0318528e-4f, 0.037005995f) : 0.0f;  // x * dq/dx
  return 0.5f * (1.0f + th) + 0.5f * x * (1.0f - th * th) * (q + dq);
}
// value and derivative together (one MUFU.TANH instead of two)
W2S_DEVINL void gelu_tanh_both(float x, float& val, float& grad) {
  const float x2 = x * x;
  const float t = fminf(x2, 25.0f);
  const float q = fmaf(fmaf(t, -3.5159264e-4f, 0.037005995f), t, 0.79750759f);
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(x * q));
  const float h = 0.5f * x;
  val = fmaf(h, th, h);
  const float dq = x2 < 25.0f ? 2.0f * x2 * fmaf(t, -7.0318528e-4f, 0.037005995f) : 0.0f;  // x * dq/dx
  grad = 0.5f * (1.0f + th) + h * (1.0f - th * th) * (q + dq);
}
// per-(sample, channel) InstanceNorm constants from fp64 sums
W2S_DEVINL void in_consts(const double* stats, int b, int C, int c, int L, float eps, float& mean, float& rstd) {
  const double s0 = stats[((size_t)b * C + c) * 2], s1 = stats[((size_t)b * C + c) * 2 + 1];
  const double m = s0 / (double)L;
  const double var = fmax(s1 / (double)L - m * m, 0.0);
  mean = (float)m;
  rstd = (float)(1.0 / sqrt(var + (double)eps));
}


}  // namespace w2s
