// Persistent, warp-specialised streaming version of the encoder conv (k=3, pad=1, stride 1|2, EPI_STATS).
//
// Same math and memory formats as conv_igemm.cuh, different execution structure.  The tile-per-CTA kernel is
// latency bound on the big C=16/32 layers (load -> transform -> MMA -> epilogue run back to back in every CTA);
// here one CTA per SM walks a contiguous range of tiles and the four stages run concurrently on different tiles:
//
//   warp 0 (1 lane)  : producer   - one cp.async.bulk (TMA, 1-D) per tile: the tile's input rows are one
//                                   contiguous byte range of the channels-last tensor -> raw ring in smem
//   warps 2+E..      : transform  - raw fp16 -> InstanceNorm (whole-night stats of the producer layer) -> GELU
//                                   [-> + residual branch -> GELU] -> fp16 (hi [+ lo]) in UMMA chunk-major layout
//   warp 1 (1 lane)  : MMA issuer - tcgen05.mma per 128-row sub-tile and tap into a double-buffered TMEM stage
//   warps 2..5       : epilogue   - tcgen05.ld, fp16 store, sum / sum-of-squares kept in registers across tiles and
//                                   flushed with fp64 atomics only when the sample changes
// Stages hand over through mbarriers (raw full, A empty, TMEM full/empty) and named barriers (transform -> producer
// "raw stage read", transform -> MMA issuer "A stage written"); weights are loaded once.
// Variants: NR = 0 (StreamCfg::DIRECT) drops the raw ring - the transform warps read global memory directly through a
// register prefetch ring (128-channel kernels); a paired launch (ConvGroup2) runs the same layer of two encoders of
// identical architecture in one grid, split in proportion to the encoders' live samples.
#pragma once
#include <cstring>

#include "conv_igemm.cuh"

namespace w2s {

// Profiling experiments (stage knock-outs, timestamps, per-role wait accounting) are compiled in only with
// -DW2S_DEBUG_KNOCKOUTS (tools/dbg_flags.sh builds such a library): in the production build ConvArgs::debug_flags is
// ignored and none of the checks below cost an instruction.
#ifdef W2S_DEBUG_KNOCKOUTS
#define W2S_DBG(p, mask) ((p).debug_flags & (mask))
#else
#define W2S_DBG(p, mask) 0
#endif
// debug_flags & 64: CTA 0 records %globaltimer at its pipeline milestones (read back with w2s_debug_timestamps)
__device__ unsigned long long g_stream_ts[16];
__device__ unsigned long long g_stream_cta_ts[2 * 512];  // debug_flags & 64: entry / exit time of every CTA
W2S_DEVINL void dbg_ts(const ConvArgs& p, int slot) {
  if (W2S_DBG(p, 64) && blockIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_stream_ts[slot] = t;
  }
}

// debug_flags & 64: cycles a role spends blocked in mbarrier waits (slot 12 MMA, 13 epilogue warp 2, 14 transform
// warp 0, 15 = total cycles of the CTA), to see which stage the pipeline is waiting for.
struct WaitClock {
  long long acc = 0;
  W2S_DEVINL void wait(const ConvArgs& p, uint64_t* bar, uint32_t parity) {
    if (W2S_DBG(p, 64)) {
      const long long t0 = clock64();
      mbar_wait(bar, parity);
      acc += clock64() - t0;
    } else {
      mbar_wait(bar, parity);
    }
  }
  W2S_DEVINL void publish(const ConvArgs& p, int slot) const {
    if (W2S_DBG(p, 64) && blockIdx.x == 0) g_stream_ts[slot] = (unsigned long long)acc;
  }
};

// warp 0 producer, 1 MMA, 2..2+E-1 epilogue, then transform.  E = 4 or 8: with 8, two warps share each TMEM lane
// quadrant (a warp may only read the quadrant warp_id % 4) and split the (column group, sub-tile) items.  Measured for
// COUT >= 64, where the epilogue is the busiest stage (93 %): no gain from 8 warps, and none from software-pipelining
// the tcgen05.ld of the next item behind the current one (register pressure eats it) - so E stays 4.  Re-measured in
// round 2 on top of the staged epilogue (a second warp per quadrant taking every other 32 x 32/64 item of the 32- and
// 64-channel kernels, 768 threads at 80 registers): same step time (6.68 vs 6.70 ms, 3 alternating rounds) - with the
// epilogue relieved, the transform warps (81 % busy) and the shared issue slots are the next limit.
constexpr int stream_epi_warps(int /*cout*/) { return 4; }
constexpr int stream_first_transform_warp(int cout) { return 2 + stream_epi_warps(cout); }
constexpr int stream_threads(int ntw, int cout) { return 32 * (stream_first_transform_warp(cout) + ntw); }

// Named-barrier hand-over (transform warps -> MMA issuer / producer): bar.arrive does not block the arriving warp and
// bar.sync parks the waiting warp in hardware until the count is reached - no polling.  ncu source view of the round-2
// kernels: 15 % of the executed warp instructions were still mbarrier polls of waiting roles (SYNCS 6.4 %, NANOSLEEP 2.9 %
// and their branches), because a parked try_wait is woken by every mbarrier event of the CTA and the transform warps
// produced 36 such events per tile.
W2S_DEVINL void named_arrive(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
W2S_DEVINL void named_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

W2S_DEVINL void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
W2S_DEVINL void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// 1-D bulk async copy global -> shared (TMA engine), completion counted in bytes on an mbarrier.
W2S_DEVINL void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// 16 consecutive channels of one output row: fp16 (2 x 16 B) or, for wide storage, fp32 (4 x 16 B).
template <bool WIDE>
W2S_DEVINL void store16(uint8_t* base, size_t elem, const float (&v)[16]) {
  if (WIDE) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint32_t w[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) w[k] = __float_as_uint(v[8 * h + k]);
      stg256(base + elem * 4 + 32 * h, w);
    }
  } else {
    const uint32_t w[8] = {pack_h2(v[0], v[1]),   pack_h2(v[2], v[3]),   pack_h2(v[4], v[5]),   pack_h2(v[6], v[7]),
                           pack_h2(v[8], v[9]),   pack_h2(v[10], v[11]), pack_h2(v[12], v[13]), pack_h2(v[14], v[15])};
    stg256(base + elem * 2, w);
  }
}

// Region stride (rows of 16 B) of the chunk-major A staging, padded so that the 8 lanes of a quarter-warp, which
// write min(8, CH*STRIDE) different (phase, chunk) regions, hit disjoint shared-memory banks.
constexpr int stream_rpad(int rp, int ch, int stride) {
  const int nreg = ch * stride < 8 ? ch * stride : 8;
  const int q = 8 / nreg;  // consecutive rows per region per quarter-warp
  int r = rp;
  while (nreg > 1 && (r % 8) != q && !(q == 1 && (r % 2) == 1)) ++r;
  return r;
}

// WIN / WOUT: the input (y and residual) / output (y and residual branch) tensors are stored as fp32 instead of fp16
// ("wide" storage of the leading blocks of deep encoders, see DESIGN.md "Numerics").
template <int CIN, int COUT, int STRIDE, int PRO, bool HAS_DS, bool SPLIT, int MT, int NR, int NA, int NTW,
          bool WIN = false, bool WOUT = false>
struct StreamCfg {
  static constexpr int CH = CIN / 8;
  // NR == 0: no raw ring - the transform warps read their 16-byte chunks straight from global memory (coalesced: a
  // tile's input rows are one contiguous byte range) through a register prefetch ring that runs one tile ahead, and
  // the shared memory of the ring goes to a second / third A stage.  Built for the 128-channel kernels, whose 96-128 KB
  // of weights left room for only ONE A stage next to a raw ring (transform and MMA of consecutive tiles serialised).
  static constexpr bool DIRECT = (NR == 0);
  static constexpr int ESZ = WIN ? 4 : 2;  // bytes per stored input element
  static constexpr int POS = 128 * MT;
  static constexpr int R = (POS - 1) * STRIDE + 3;            // input rows per tile (with halo)
  static constexpr int RP = stream_rpad((R + STRIDE - 1) / STRIDE, CH, STRIDE);  // rows per stride phase (padded)
  static constexpr int THREADS = stream_threads(NTW, COUT);
  static constexpr int EPI_WARPS = stream_epi_warps(COUT);
  static constexpr int FIRST_TW = stream_first_transform_warp(COUT);
  // raw ring entry: [y rows (fp16)] [residual rows (fp16) | raw-signal floats for the block-0 fusion modes]
  static constexpr int XN = (PRO == PRO_FIR) ? R + 12 : (PRO == PRO_NORM_RES_X) ? 2 * R + 12 : 0;  // staged x floats
  static constexpr int RAW_ONE = (PRO == PRO_FIR) ? 0 : (R * CIN * ESZ + 127) / 128 * 128;
  static constexpr int RAW_X = (XN * 4 + 127) / 128 * 128;
  static constexpr int RAW_BYTES = RAW_ONE * (PRO == PRO_NORM_RES ? 2 : 1) + RAW_X;
  static constexpr int A_ONE = STRIDE * CH * RP * 16;
  static constexpr int A_BYTES = A_ONE * (SPLIT ? 2 : 1);
  static constexpr int B_ONE = (3 + (HAS_DS ? 1 : 0)) * CH * COUT * 16;
  static constexpr int B_BYTES = B_ONE * (SPLIT ? 2 : 1);
  static constexpr int STAGE_COLS = MT * COUT * (HAS_DS ? 2 : 1);
  static constexpr int TMEM_COLS = (2 * STAGE_COLS <= 32) ? 32 : (2 * STAGE_COLS <= 64) ? 64 : (2 * STAGE_COLS <= 128) ? 128 : (2 * STAGE_COLS <= 256) ? 256 : 512;
  static constexpr int CTL_BYTES = 768;  // mbarriers + TMEM slot (first 256 B), live-sample lists of the two groups (256 B each)
  static constexpr int SMEM_BASE = NR * RAW_BYTES + NA * A_BYTES + B_BYTES + CTL_BYTES;
  // per-thread statistics accumulators across tiles for COUT = 16 (and for the 32-channel conv1 kernels, whose epilogue
  // also drains the residual-branch accumulator: measured faster)
  // (re-measured against the staged epilogue with 14 instead of 10 transform warps, which the lower register count
  // would allow: 16 -> 32 conv1 273 -> 354 us, 32 -> 32 conv1 219 -> 237 us per paired launch - slower)
  static constexpr bool REG_STATS = (COUT <= 16) || (COUT <= 32 && HAS_DS);
  // Staged epilogue (all other fp16-output kernels, where shared memory allows): each epilogue warp transposes its
  // 32 rows through a private, XOR-swizzled staging buffer, so that (i) global stores are full 128-byte lines written
  // by 8 adjacent lanes instead of 32 scattered 32-byte sectors per instruction, and (ii) every lane keeps a fixed set
  // of 8 channels, whose sum / sum of squares live in registers across tiles - no per-tile warp butterflies (they were
  // ~60 shuffles per 16 channels per tile, the busiest stage of the 64/128-channel kernels).
  static constexpr int SEG = COUT < 64 ? COUT : 64;  // channels per staged row segment (64 or 128 bytes)
  static constexpr int STAGE_WARP_BYTES = 32 * SEG * 2;
  static constexpr bool STAGED = !REG_STATS && !WOUT && (SMEM_BASE + 4 * STAGE_WARP_BYTES <= 232448);
  static constexpr int SMEM_BYTES = SMEM_BASE + (STAGED ? 4 * STAGE_WARP_BYTES : 0);
  static_assert(2 * STAGE_COLS <= 512, "TMEM budget");
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
  static_assert((NTW * 32) % CH == 0, "fixed channel chunk per transform thread");
  static_assert(!DIRECT || ((PRO == PRO_NORM || PRO == PRO_NORM_RES) && !WIN), "direct-from-global transform: fp16 PRO_NORM[_RES] only");
  // direct mode: 16-byte chunks per transform thread and tile, and the depth of the register prefetch ring
  static constexpr int NIT = (R * CH + NTW * 32 - 1) / (NTW * 32);
  static constexpr int PF = NIT <= 5 ? NIT : (NIT + 1) / 2;
};

template <int CIN, int COUT, int STRIDE, int PRO, bool HAS_DS, bool SPLIT, int MT, int NR, int NA, int NTW, bool WIN, bool WOUT>
__global__ void __launch_bounds__(stream_threads(NTW, COUT), (stream_threads(NTW, COUT) <= 384 ? 2 : 1))
conv_stream_kernel(const ConvArgs pa, const ConvGroup2 pb, int tiles_per_sample, int total_tiles) {
  // group of this CTA and the argument block it works on (scalars stay kernel-parameter constants, pointers are selected)
  // (the group of a CTA is decided after the set-up barrier, from the two groups' live-sample counts; each role then
  // overrides only the pointers it uses, inside its own branch: keeps the selects out of the other roles' registers)
  constexpr bool kPairable = stream_pairable(COUT, HAS_DS);
  const bool paired = kPairable && pb.ngroups > 1;
  ConvArgs p = pa;
  using Cfg = StreamCfg<CIN, COUT, STRIDE, PRO, HAS_DS, SPLIT, MT, NR, NA, NTW, WIN, WOUT>;
  constexpr int ESZ = Cfg::ESZ;
  constexpr int kStreamThreads = Cfg::THREADS;
  constexpr int kStreamTransformWarps = NTW;
  constexpr int kStreamFirstTransformWarp = Cfg::FIRST_TW;
  constexpr int EPI_SPLIT = Cfg::EPI_WARPS / 4;  // epilogue warps per TMEM lane quadrant
  constexpr int CH = Cfg::CH, POS = Cfg::POS, R = Cfg::R, RP = Cfg::RP;
  constexpr int KSTEPS = CIN / 16;
  constexpr int NCG = COUT / 16;
  constexpr uint32_t IDESC = umma_idesc_f16(128, COUT, false);
  constexpr bool REG_STATS = Cfg::REG_STATS;
  constexpr bool STAGED = Cfg::STAGED;
  // named barriers: ids 1 .. NA = "A stage written" (transform -> MMA issuer), NA+1 .. NA+NR = "raw stage read"
  // (transform -> producer); each is joined by the NTW transform warps (bar.arrive) and the one waiting warp (bar.sync)
  constexpr int kNamedCount = 32 * (NTW + 1);
  static_assert(NA + NR < 16, "named barrier ids");

  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* sRaw = smem;
  uint8_t* sA = sRaw + NR * Cfg::RAW_BYTES;
  uint8_t* sB = sA + NA * Cfg::A_BYTES;
  uint8_t* sCtl = sB + Cfg::B_BYTES;
  uint64_t* raw_full = reinterpret_cast<uint64_t*>(sCtl);
  uint64_t* a_empty = raw_full + NR;
  uint64_t* t_full = a_empty + NA;
  uint64_t* t_empty = t_full + 2;
  uint64_t* w_full = t_empty + 2;  // weights landed in sB (one bulk-copy transaction group per CTA)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_full + 1);
  uint8_t* sStage = sCtl + Cfg::CTL_BYTES;  // STAGED: 4 warp-private staging buffers
  (void)sStage;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // Samples without this signal (row_mask) are compacted away before the tiles are split over the CTAs, so that masked
  // nights cost nothing and the remaining work stays balanced (training with the modality masker, inference with
  // missing signals).  sLive[i] = i-th live sample; batches larger than the list fall back to skipping tile by tile.
  constexpr int kMaxLive = 120;
  uint16_t* sLive0 = reinterpret_cast<uint16_t*>(sCtl + 256);
  uint16_t* sLive1 = reinterpret_cast<uint16_t*>(sCtl + 512);  // second group of a paired launch
  int* sNLive = reinterpret_cast<int*>(sCtl + 256 + 2 * kMaxLive);  // [0] group 0; group 1 at the same place of its block
  int* sNLive1 = reinterpret_cast<int*>(sCtl + 512 + 2 * kMaxLive);
  const int n_samples = total_tiles / tiles_per_sample;
  const bool compact = pa.row_mask != nullptr && n_samples <= kMaxLive;

  // ---------------- one-time setup ----------------
  if (tid == 0) dbg_ts(p, 0);
  if (W2S_DBG(p, 64) && tid == 0 && blockIdx.x < 512) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_stream_cta_ts[2 * blockIdx.x] = t;
  }
  if (warp == 0) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  if (tid == 0) dbg_ts(p, 1);
  if (tid == 32) {
    for (int s = 0; s < NR; ++s) mbar_init(&raw_full[s], 1);
    for (int s = 0; s < NA; ++s) mbar_init(&a_empty[s], 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&t_full[s], 1);
      mbar_init(&t_empty[s], Cfg::EPI_WARPS);
    }
    mbar_init(w_full, 1);
    fence_mbar_init();
  }
  if (compact && warp == 2) {
    const int n = build_live_list(pa.row_mask, n_samples, sLive0, lane);
    if (lane == 0) *sNLive = n;
  }
  if (compact && paired && warp == 3) {
    const int n = build_live_list(pb.row_mask, n_samples, sLive1, lane);
    if (lane == 0) *sNLive1 = n;
  }
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  // Paired launch: the grid is split between the two encoders in proportion to their live samples (the modality masks
  // of the two signals differ: a night without PPG costs the ECG + PPG launch nothing on the PPG side, and the CTAs it
  // would have had work on ECG instead); without compaction, half each.
  int ctas0 = (int)gridDim.x;
  if (paired) {
    ctas0 = (int)gridDim.x >> 1;
    if (compact) {
      const int n0 = *sNLive, n1 = *sNLive1;
      if (n0 != n1) {  // (equal counts: half each, nothing to compute; 32-bit: gridDim.x * n0 <= 296 * 120)
        ctas0 = (int)(((unsigned)gridDim.x * (unsigned)n0 + ((unsigned)(n0 + n1) >> 1)) / (unsigned)(n0 + n1));
        if (n0 > 0 && ctas0 < 1) ctas0 = 1;
        if (n1 > 0 && ctas0 > (int)gridDim.x - 1) ctas0 = (int)gridDim.x - 1;
      }
    }
  }
  const bool grp1 = paired && (int)blockIdx.x >= ctas0;
  const int cta = grp1 ? (int)blockIdx.x - ctas0 : (int)blockIdx.x;
  const int nctas = grp1 ? (int)gridDim.x - ctas0 : ctas0;
  if (grp1) p.row_mask = pb.row_mask;
  const uint16_t* sLive = grp1 ? sLive1 : sLive0;
  const int live_tiles = compact ? (grp1 ? *sNLive1 : *sNLive) * tiles_per_sample : total_tiles;
  const int tile_begin = (int)((long long)cta * live_tiles / nctas);
  const int tile_end = (int)((long long)(cta + 1) * live_tiles / nctas);
  // Position of a tile as (entry of the sample list, tile inside the sample), advanced incrementally: no division in
  // the per-tile loops of the four roles.
  struct TilePos {
    int s, r;
  };
  const TilePos pos0 = {tile_begin / tiles_per_sample, tile_begin % tiles_per_sample};
  auto advance = [&](TilePos& t) {
    if (++t.r == tiles_per_sample) {
      t.r = 0;
      ++t.s;
    }
  };
  // sample of a tile position; false = masked sample (only possible without compaction)
  auto sample_of = [&](const TilePos& t, int& b) {
    b = compact ? (int)sLive[t.s] : t.s;
    return compact || p.row_mask == nullptr || !p.row_mask[b];
  };

  // ======================================================================================================
  if (warp == 0) {
    // ---------------- producer (whole warp runs the loop; one elected lane issues) ----------------
    if (grp1) {
      p.in = pb.in; p.in_res = pb.in_res; p.x_raw = pb.x_raw; p.w = pb.w; p.w_ds = pb.w_ds;
    }
    {
      // weights -> smem once per CTA (hi [, lo] blocks; the 1x1 branch after the taps): plain bulk copies of the packed
      // layout, off every other role's critical path (only the MMA issuer waits for them)
      if (tile_begin < tile_end && elect_one()) {  // (a CTA without tiles must not leave a copy in flight when it exits)
        constexpr uint32_t wbytes = 3u * CH * COUT * 16u, dbytes = (uint32_t)CH * COUT * 16u;
        mbar_arrive_expect_tx(w_full, (wbytes + (HAS_DS ? dbytes : 0u)) * (SPLIT ? 2u : 1u));
        const uint8_t* gw = reinterpret_cast<const uint8_t*>(p.w);
        bulk_g2s(sB, gw, wbytes, w_full);
        if (SPLIT) bulk_g2s(sB + Cfg::B_ONE, gw + wbytes, wbytes, w_full);
        if (HAS_DS) {
          const uint8_t* gd = reinterpret_cast<const uint8_t*>(p.w_ds);
          bulk_g2s(sB + wbytes, gd, dbytes, w_full);
          if (SPLIT) bulk_g2s(sB + Cfg::B_ONE + wbytes, gd + dbytes, dbytes, w_full);
        }
      }
      __syncwarp();
      int s = 0, n_issued = 0;
      const long long cta_t0 = clock64();
      TilePos tp = pos0;
      for (int tile = tile_begin; tile < (Cfg::DIRECT ? tile_begin : tile_end); ++tile, advance(tp)) {
        int b;
        if (!sample_of(tp, b)) continue;
        const int o0 = tp.r * POS;
        const int i0 = o0 * STRIDE - 1;
        const int lo = i0 < 0 ? 0 : i0;
        const int hi = (i0 + R < p.L_in) ? i0 + R : p.L_in;
        const uint32_t nbytes = (PRO == PRO_FIR) ? 0u : (uint32_t)(hi - lo) * CIN * ESZ;
        // raw-signal window of the block-0 fusion modes: x[xs0, xs0 + Cfg::XN) clipped to the sample, 16-B aligned
        //   PRO_FIR        : conv1 needs x[i - 1 .. i + 1] for the staged rows i = i0 .. i0 + R - 1
        //   PRO_NORM_RES_X : the residual branch needs x[2 i]
        const int xs0 = (PRO == PRO_FIR) ? ((i0 - 1) & ~3) : ((2 * i0) & ~3);  // floor to a multiple of 4 (also < 0)
        const int xlo = xs0 < 0 ? 0 : xs0;
        int xhi = xs0 + Cfg::XN;
        xhi = (xhi > p.T_raw ? p.T_raw : xhi) & ~3;
        const uint32_t xbytes = (Cfg::XN > 0 && xhi > xlo) ? (uint32_t)(xhi - xlo) * 4 : 0u;
        if (n_issued >= NR) named_sync(1 + NA + s, kNamedCount);  // (the first NR fills find the ring empty)
        ++n_issued;
        uint8_t* dst = sRaw + s * Cfg::RAW_BYTES + (size_t)(lo - i0) * CIN * ESZ;
        const size_t goff = ((size_t)b * p.L_in + lo) * CIN * ESZ;  // byte offset
        if (elect_one()) {
          mbar_arrive_expect_tx(&raw_full[s], nbytes * (PRO == PRO_NORM_RES ? 2u : 1u) + xbytes);
          if (PRO != PRO_FIR) bulk_g2s(dst, reinterpret_cast<const uint8_t*>(p.in) + goff, nbytes, &raw_full[s]);
          if (PRO == PRO_NORM_RES)
            bulk_g2s(dst + Cfg::RAW_ONE, reinterpret_cast<const uint8_t*>(p.in_res) + goff, nbytes, &raw_full[s]);
          if (Cfg::XN > 0 && xbytes > 0)
            bulk_g2s(sRaw + s * Cfg::RAW_BYTES + Cfg::RAW_ONE + (size_t)(xlo - xs0) * 4,
                     p.x_raw + (size_t)b * p.T_raw + xlo, xbytes, &raw_full[s]);
        }
        __syncwarp();
        if (++s == NR) s = 0;
      }
      if (lane == 0 && W2S_DBG(p, 64) && blockIdx.x == 0) g_stream_ts[15] = (unsigned long long)(clock64() - cta_t0);
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer (warp-uniform loop; one elected lane issues) ----------------
    {
      int as = 0, ts = 0;
      uint32_t tph = 0;
      WaitClock wc;
      constexpr uint32_t lbo_a = RP * 16, lbo_b = COUT * 16;
      // descriptors = (stage / operand base) + compile-time offset: one integer add per operand on the issuing thread
      constexpr uint32_t DHI = umma_desc_hi(128);
      const uint32_t b_lo0 = umma_desc_lo(smem_u32(sB), lbo_b);
      const uint32_t a_lo_first = umma_desc_lo(smem_u32(sA), lbo_a);
      uint32_t a_lo0 = a_lo_first;
      TilePos tp = pos0;
      if (tile_begin < tile_end) mbar_wait(w_full, 0);
      for (int tile = tile_begin; tile < tile_end; ++tile, advance(tp)) {
        int b;
        if (!sample_of(tp, b)) continue;
        named_sync(1 + as, kNamedCount);
        wc.wait(p, &t_empty[ts], tph ^ 1);
        tc_fence_after_sync();
        const uint32_t d_base = tmem_base + ts * Cfg::STAGE_COLS;
        if (elect_one()) {
#pragma unroll
        for (int j = 0; j < MT; ++j) {
#pragma unroll
          for (int t = 0; t < 3; ++t) {
            const int phase = t & (STRIDE - 1);
            const int rowoff = t / STRIDE + j * 128;
#pragma unroll
            for (int kk = 0; kk < KSTEPS; ++kk) {
              const uint32_t a_off = (uint32_t)((phase * CH + 2 * kk) * RP + rowoff);       // in 16-byte units
              const uint32_t b_off = (uint32_t)((t * CH + 2 * kk) * COUT);
              const uint64_t da = umma_desc(a_lo0 + a_off, DHI);
              const uint64_t db = umma_desc(b_lo0 + b_off, DHI);
              if (!W2S_DBG(p, 2)) umma_f16(d_base + j * COUT, da, db, IDESC, (t > 0 || kk > 0) ? 1u : 0u);
              if (SPLIT && !W2S_DBG(p, 3)) {
                if (!W2S_DBG(p, 128) && !(CIN == 32 && W2S_DBG(p, 512)))
                  umma_f16(d_base + j * COUT, umma_desc(a_lo0 + (Cfg::A_ONE >> 4) + a_off, DHI), db, IDESC, 1u);
                if (!W2S_DBG(p, 256) && !(CIN == 32 && W2S_DBG(p, 1024)))
                  umma_f16(d_base + j * COUT, da, umma_desc(b_lo0 + (Cfg::B_ONE >> 4) + b_off, DHI), IDESC, 1u);
              }
            }
          }
          if (HAS_DS) {  // 1x1 stride-2 residual branch on the centre tap rows (STRIDE == 1 here)
            const int rowoff = 1 + j * 128;
#pragma unroll
            for (int kk = 0; kk < KSTEPS; ++kk) {
              const uint32_t a_off = (uint32_t)((2 * kk) * RP + rowoff);
              const uint32_t b_off = (uint32_t)((3 * CH + 2 * kk) * COUT);
              const uint64_t da = umma_desc(a_lo0 + a_off, DHI);
              const uint64_t db = umma_desc(b_lo0 + b_off, DHI);
              umma_f16(d_base + (MT + j) * COUT, da, db, IDESC, kk > 0 ? 1u : 0u);
              if (SPLIT) {
                if (!W2S_DBG(p, 128))
                  umma_f16(d_base + (MT + j) * COUT, umma_desc(a_lo0 + (Cfg::A_ONE >> 4) + a_off, DHI), db, IDESC, 1u);
                if (!W2S_DBG(p, 256))
                  umma_f16(d_base + (MT + j) * COUT, da, umma_desc(b_lo0 + (Cfg::B_ONE >> 4) + b_off, DHI), IDESC, 1u);
              }
            }
          }
        }
        umma_commit(&a_empty[as]);  // A stage reusable once these MMAs have read it
        umma_commit(&t_full[ts]);   // accumulators ready for the epilogue
        }
        __syncwarp();
        a_lo0 += Cfg::A_BYTES >> 4;
        if (++as == NA) {
          as = 0;
          a_lo0 = a_lo_first;
        }
        if (++ts == 2) {
          ts = 0;
          tph ^= 1;
        }
      }
      if (lane == 0) wc.publish(p, 12);
    }
  } else if (warp < kStreamFirstTransformWarp) {
    // ---------------- epilogue (warps 2..5 -> TMEM lane quadrants 2,3,0,1) ----------------
    if (grp1) {
      p.out = pb.out; p.out_ds = pb.out_ds; p.out_stats = pb.out_stats;
    }
    if constexpr (STAGED) {
      static_assert(Cfg::EPI_WARPS == 4, "one epilogue warp per TMEM lane quadrant");
      constexpr int SEG = Cfg::SEG, SEGB = SEG * 2;
      constexpr int LPR = SEGB / 16;   // lanes per row segment in the copy-out (4 or 8)
      constexpr int RPI = 32 / LPR;    // rows per copy-out instruction (8 or 4)
      constexpr int NSEG = COUT / SEG;
      const int quad = warp & 3;
      const uint32_t t_lane = (uint32_t)(quad * 32) << 16;
      const uint32_t stg = smem_u32(sStage + (warp - 2) * Cfg::STAGE_WARP_BYTES);
      const int crow = lane / LPR, cchunk = lane % LPR;  // this lane's role in the copy-out: row in group, 16-B chunk
      // 16-B chunk c of staged row r sits at r * SEGB + ((c ^ swz(r)) * 16): conflict-free for the row-per-lane writes
      // (8 rows x same chunk per quarter-warp) and for the row-segment reads (LPR lanes x consecutive chunks)
      auto swz = [](int r) { return SEGB == 128 ? (r & 7) : ((r >> 1) & 3); };
      int ts = 0;
      uint32_t tph = 0;
      int cur_b = -1;
      WaitClock wc;
      float2 ssum[NSEG][4], ssq[NSEG][4];  // this lane's 8 channels of each segment, over every row it copies out
#pragma unroll
      for (int sg = 0; sg < NSEG; ++sg)
#pragma unroll
        for (int k = 0; k < 4; ++k) ssum[sg][k] = ssq[sg][k] = make_float2(0.0f, 0.0f);
      auto flush = [&](int b) {
        if (b < 0) return;
#pragma unroll
        for (int sg = 0; sg < NSEG; ++sg) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float v[4] = {ssum[sg][k].x, ssum[sg][k].y, ssq[sg][k].x, ssq[sg][k].y};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
#pragma unroll
              for (int off = LPR; off < 32; off <<= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], off);
            }
            if (lane < LPR) {
              const int c = sg * SEG + cchunk * 8 + 2 * k;
              atomicAdd(&p.out_stats[((size_t)b * COUT + c) * 2 + 0], (double)v[0]);
              atomicAdd(&p.out_stats[((size_t)b * COUT + c + 1) * 2 + 0], (double)v[1]);
              atomicAdd(&p.out_stats[((size_t)b * COUT + c) * 2 + 1], (double)v[2]);
              atomicAdd(&p.out_stats[((size_t)b * COUT + c + 1) * 2 + 1], (double)v[3]);
            }
            ssum[sg][k] = ssq[sg][k] = make_float2(0.0f, 0.0f);
          }
        }
      };
      // TMEM columns [col, col + SEG) of this warp's 32 lanes -> staging (lane = row).  All loads of the segment are
      // issued before the single tcgen05.wait::ld: the round trip of a TMEM load while the MMA unit is accumulating
      // into the other stage is several hundred cycles, and it used to be paid once per 16 columns.
      auto stage_in = [&](uint32_t taddr) {
        uint32_t r[SEG];
#pragma unroll
        for (int q = 0; q < SEG / 32; ++q) tmem_ld32(taddr + q * 32, r + q * 32);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < SEG / 8; ++c) {
          const uint4 w = make_uint4(pack_h2(__uint_as_float(r[8 * c]), __uint_as_float(r[8 * c + 1])),
                                     pack_h2(__uint_as_float(r[8 * c + 2]), __uint_as_float(r[8 * c + 3])),
                                     pack_h2(__uint_as_float(r[8 * c + 4]), __uint_as_float(r[8 * c + 5])),
                                     pack_h2(__uint_as_float(r[8 * c + 6]), __uint_as_float(r[8 * c + 7])));
          sts128(stg + lane * SEGB + ((c ^ swz(lane)) * 16), w);
        }
      };
      TilePos tp = pos0;
      for (int tile = tile_begin; tile < tile_end; ++tile, advance(tp)) {
        int b;
        if (!sample_of(tp, b)) continue;
        if (b != cur_b) {
          flush(cur_b);
          cur_b = b;
        }
        const int o0 = tp.r * POS;
        wc.wait(p, &t_full[ts], tph);
        tc_fence_after_sync();
        const uint32_t d_base = tmem_base + ts * Cfg::STAGE_COLS + t_lane;
        uint8_t* outb = reinterpret_cast<uint8_t*>(p.out) + (size_t)b * p.L_out * COUT * 2;
#pragma unroll 1
        for (int j = 0; j < MT; ++j) {
          const int obase = o0 + j * 128 + quad * 32;
#pragma unroll
          for (int sg = 0; sg < NSEG; ++sg) {
            if (!W2S_DBG(p, 16)) stage_in(d_base + j * COUT + sg * SEG);
            __syncwarp();
            if (!HAS_DS && j == MT - 1 && sg == NSEG - 1) {  // accumulators drained: hand the TMEM stage back early
              tc_fence_before_sync();
              if (lane == 0) mbar_arrive(&t_empty[ts]);
            }
#pragma unroll
            for (int it = 0; it < 32 / RPI; ++it) {
              const int r = it * RPI + crow;
              const int o = obase + r;
              const uint4 val = lds128(stg + r * SEGB + ((cchunk ^ swz(r)) * 16));
              if (o < p.L_out && !W2S_DBG(p, 8)) {
                *reinterpret_cast<uint4*>(outb + ((size_t)o * COUT + sg * SEG + cchunk * 8) * 2) = val;
                const uint32_t w4[4] = {val.x, val.y, val.z, val.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const float2 f = unpack_h2(w4[k]);
                  ssum[sg][k] = __fadd2_rn(ssum[sg][k], f);
                  ssq[sg][k] = __ffma2_rn(f, f, ssq[sg][k]);
                }
              }
            }
            __syncwarp();
          }
        }
        if (HAS_DS) {
          uint8_t* dsb = reinterpret_cast<uint8_t*>(p.out_ds) + (size_t)b * (p.L_out >> 1) * COUT * 2;
#pragma unroll 1
          for (int j = 0; j < MT; ++j) {
            const int obase = o0 + j * 128 + quad * 32;  // even
#pragma unroll
            for (int sg = 0; sg < NSEG; ++sg) {
              stage_in(d_base + (MT + j) * COUT + sg * SEG);
              __syncwarp();
              if (j == MT - 1 && sg == NSEG - 1) {
                tc_fence_before_sync();
                if (lane == 0) mbar_arrive(&t_empty[ts]);
              }
#pragma unroll
              for (int it = 0; it < 16 / RPI; ++it) {  // even rows only: the 1x1 branch has stride 2
                const int r = 2 * (it * RPI + crow);
                const int o = obase + r;
                const uint4 val = lds128(stg + r * SEGB + ((cchunk ^ swz(r)) * 16));
                if (o < (p.L_out & ~1))  // out_ds has L_out / 2 rows (rounded down)
                  *reinterpret_cast<uint4*>(dsb + ((size_t)(o >> 1) * COUT + sg * SEG + cchunk * 8) * 2) = val;
              }
              __syncwarp();
            }
          }
        }
        if (++ts == 2) {
          ts = 0;
          tph ^= 1;
        }
      }
      if (warp == 2 && lane == 0) wc.publish(p, 13);
      flush(cur_b);
    } else {
    const int quad = warp & 3;
    const int epi_half = (warp - 2) >> 2;  // which share of the (column group, sub-tile) items this warp takes
    const uint32_t t_lane = (uint32_t)(quad * 32) << 16;
    int ts = 0;
    uint32_t tph = 0;
    int cur_b = -1;
    WaitClock wc;
    constexpr int NACC = REG_STATS ? NCG * 16 : NCG;
    float acc[NACC], acc2[NACC];
#pragma unroll
    for (int k = 0; k < NACC; ++k) acc[k] = acc2[k] = 0.0f;

    auto flush = [&](int b) {
      if (b < 0) return;
#pragma unroll
      for (int cg = 0; cg < NCG; ++cg) {
        float s0, s1;
        if (REG_STATS) {
          butterfly16(&acc[cg * 16], lane);
          butterfly16(&acc2[cg * 16], lane);
          s0 = acc[cg * 16];
          s1 = acc2[cg * 16];
        } else {
          s0 = acc[cg];
          s1 = acc2[cg];
        }
        if ((lane & 1) == 0) {
          const int c = cg * 16 + butterfly16_channel(lane);
          atomicAdd(&p.out_stats[((size_t)b * COUT + c) * 2 + 0], (double)s0);
          atomicAdd(&p.out_stats[((size_t)b * COUT + c) * 2 + 1], (double)s1);
        }
      }
#pragma unroll
      for (int k = 0; k < NACC; ++k) acc[k] = acc2[k] = 0.0f;
    };

    TilePos tp = pos0;
    for (int tile = tile_begin; tile < tile_end; ++tile, advance(tp)) {
      int b;
      if (!sample_of(tp, b)) continue;
      if (b != cur_b) {
        flush(cur_b);
        cur_b = b;
      }
      const int o0 = tp.r * POS;
      wc.wait(p, &t_full[ts], tph);
      tc_fence_after_sync();
      if (warp == 2 && lane == 0 && tile == tile_begin) dbg_ts(p, 6);
      const uint32_t d_base = tmem_base + ts * Cfg::STAGE_COLS + t_lane;
      uint8_t* outb = reinterpret_cast<uint8_t*>(p.out) + (size_t)b * p.L_out * COUT * (WOUT ? 4 : 2);
#pragma unroll
      for (int cg = 0; cg < NCG; ++cg) {
        float ps[16], pq[16];
        if (!REG_STATS) {
#pragma unroll
          for (int k = 0; k < 16; ++k) ps[k] = pq[k] = 0.0f;
        }
#pragma unroll 1
        for (int j = 0; j < MT; ++j) {
          float v[16];
          if (EPI_SPLIT > 1 && ((cg * MT + j) % EPI_SPLIT) != epi_half) continue;
          if (W2S_DBG(p, 16)) continue;
          tmem_ld16(d_base + j * COUT + cg * 16, v);
          const int o = o0 + j * 128 + quad * 32 + lane;
          if (o < p.L_out && !(W2S_DBG(p, 8) && v[0] != 123.456f)) {
            store16<WOUT>(outb, (size_t)o * COUT + cg * 16, v);
#pragma unroll
            for (int k = 0; k < 16; k += 2) {  // packed fp32x2: one FADD2 + one FFMA2 per channel pair
              const float2 vv = make_float2(v[k], v[k + 1]);
              float* s = REG_STATS ? &acc[cg * 16 + k] : &ps[k];
              float* q = REG_STATS ? &acc2[cg * 16 + k] : &pq[k];
              const float2 ns = __fadd2_rn(make_float2(s[0], s[1]), vv);
              const float2 nq = __ffma2_rn(vv, vv, make_float2(q[0], q[1]));
              s[0] = ns.x;
              s[1] = ns.y;
              q[0] = nq.x;
              q[1] = nq.y;
            }
          }
        }
        if (!REG_STATS) {
          butterfly16(ps, lane);
          butterfly16(pq, lane);
          acc[cg] += ps[0];
          acc2[cg] += pq[0];
        }
      }
      if (HAS_DS) {
        uint8_t* dsb = reinterpret_cast<uint8_t*>(p.out_ds) + (size_t)b * (p.L_out >> 1) * COUT * (WOUT ? 4 : 2);
#pragma unroll 1
        for (int j = 0; j < MT; ++j) {
          const int o = o0 + j * 128 + quad * 32 + lane;
#pragma unroll
          for (int cg = 0; cg < NCG; ++cg) {
            float v[16];
            if (EPI_SPLIT > 1 && ((cg * MT + j) % EPI_SPLIT) != epi_half) continue;
            tmem_ld16(d_base + (MT + j) * COUT + cg * 16, v);
            if (o < (p.L_out & ~1) && (o & 1) == 0) {  // out_ds has L_out / 2 rows (rounded down)
              store16<WOUT>(dsb, (size_t)(o >> 1) * COUT + cg * 16, v);
            }
          }
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&t_empty[ts]);
      if (++ts == 2) {
        ts = 0;
        tph ^= 1;
      }
    }
    if (warp == 2 && lane == 0) {
      dbg_ts(p, 7);
      wc.publish(p, 13);
    }
    flush(cur_b);
    if (warp == 2 && lane == 0) dbg_ts(p, 8);
    }
  } else {
    // ---------------- transform warps ----------------
    if (grp1) {
      p.in_stats = pb.in_stats; p.w_first = pb.w_first; p.w_first_ds = pb.w_first_ds;
      if (Cfg::DIRECT) {
        p.in = pb.in; p.in_res = pb.in_res;
      }
    }
    const int tt = tid - kStreamFirstTransformWarp * 32;  // 0..255
    constexpr int NTT = kStreamTransformWarps * 32;
    const int cch = tt & (CH - 1);
    int rs = 0, as = 0;
    uint32_t rph = 0, aph = 0;
    int cur_b = -1;
    WaitClock wc_raw, wc_a;
    float2 sc[4], sh[4];  // per-channel scale / shift of this thread's 8 channels, as fp32x2 pairs
    float2 fws[4][3];     // PRO_FIR: conv1 taps pre-multiplied by the per-sample InstanceNorm scale
    float2 fw[4][3];      // block-0 fusion modes: conv1 taps (PRO_FIR) / downsample weight in [.][0] (PRO_NORM_RES_X)
    if (PRO == PRO_NORM_RES_X) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int c = cch * 8 + 2 * q;
        fw[q][0] = make_float2(__ldg(p.w_first_ds + c), __ldg(p.w_first_ds + c + 1));
      }
    }
    // per-sample constants of this thread's 8 channels
    auto load_consts = [&](int b) {
      const double inv_len = 1.0 / (double)p.L_in;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int c = cch * 8 + k;
        const double s0 = p.in_stats[((size_t)b * CIN + c) * 2 + 0];
        const double s1 = p.in_stats[((size_t)b * CIN + c) * 2 + 1];
        const double mean = s0 * inv_len;
        const double var = fmax(s1 * inv_len - mean * mean, 0.0);
        // mean / variance need fp64 (sumsq / L - mean^2 cancels); the reciprocal square root does not
        const float rstd = 1.0f / sqrtf((float)(var + (double)p.in_eps));
        if (k & 1) {
          sc[k >> 1].y = rstd;
          sh[k >> 1].y = (float)(-mean) * rstd;
        } else {
          sc[k >> 1].x = rstd;
          sh[k >> 1].x = (float)(-mean) * rstd;
        }
      }
      if (PRO == PRO_FIR) {  // taps re-read (L1/L2 hits) on a sample change instead of living in registers
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int c = cch * 8 + 2 * q;
#pragma unroll
          for (int t = 0; t < 3; ++t)
            fws[q][t] = __fmul2_rn(make_float2(__ldg(p.w_first + c * 3 + t), __ldg(p.w_first + (c + 1) * 3 + t)), sc[q]);
        }
      }
    };
    // per-tile state read by the chunk transform below
    int i0 = 0, xs0 = 0;
    uint32_t adst = 0;
    const float* xraw = nullptr;  // staged x window (block-0 fusion modes)
    bool x_interior = false;      // whole x window inside the sample
    auto xat = [&](int j) -> float {  // x[j] of this sample with conv1's zero padding and the -inf -> 0 rule
      if (!x_interior && (j < 0 || j >= p.T_raw)) return 0.0f;
      const float v = xraw[j - xs0];
      return isinf(v) ? 0.0f : v;
    };
    auto fin = [](float v) { return isinf(v) ? 0.0f : v; };  // the reference's -inf -> 0 rule, element-wise
    // Offset (bytes) of input row u in a chunk column of the A stage.  The row index of a thread's k-th chunk of a
    // tile is tt / CH + k * NTT / CH, so on interior tiles every offset is a per-thread constant plus a compile-time one.
    auto soff_of = [](int u) { return (uint32_t)((u & (STRIDE - 1)) * CH * RP + u / STRIDE) * 16; };
    // 8 channels of one input row (y [, y2]: stored conv output, r [, r2]: residual branch; xm / x0 / xp: raw-signal
    // samples of the block-0 fusion modes, -inf already replaced) -> activated fp16 operand chunk(s) at dst in the A stage
    auto act = [&](bool valid, float xm, float x0, float xp, const uint4& y, const uint4& y2, const uint4& r,
                   const uint4& r2, uint32_t dst) {
      uint4 o = make_uint4(0u, 0u, 0u, 0u), olo = make_uint4(0u, 0u, 0u, 0u);
      if (valid) {
        const uint32_t yy[8] = {y.x, y.y, y.z, y.w, y2.x, y2.y, y2.z, y2.w};
        const uint32_t rr[8] = {r.x, r.y, r.z, r.w, r2.x, r2.y, r2.z, r2.w};
        auto pair = [&](const uint32_t (&w)[8], int q) -> float2 {  // channels 2q, 2q+1 of the 8 as fp32
          return WIN ? make_float2(__uint_as_float(w[2 * q]), __uint_as_float(w[2 * q + 1])) : unpack_h2(w[q]);
        };
        uint32_t* oo = reinterpret_cast<uint32_t*>(&o);
        uint32_t* ol = reinterpret_cast<uint32_t*>(&olo);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float2 yv;
          float2 a;
          if (PRO == PRO_FIR) {
            // conv1 of block 0 recomputed in fp32 (never stored, never rounded); the InstanceNorm scale is folded
            // into the taps (fws = w * rstd), the shift is the FMA addend: 3 packed FMAs give x_hat directly
            a = __ffma2_rn(fws[q][2], make_float2(xp, xp),
                           __ffma2_rn(fws[q][1], make_float2(x0, x0), __ffma2_rn(fws[q][0], make_float2(xm, xm), sh[q])));
          } else {
            yv = pair(yy, q);
            a = __ffma2_rn(yv, sc[q], sh[q]);
          }
          if (!W2S_DBG(p, 4)) a = gelu_fast2(a);
          if (PRO == PRO_NORM_RES) a = gelu_fast2(__fadd2_rn(a, pair(rr, q)));
          if (PRO == PRO_NORM_RES_X) a = gelu_fast2(__ffma2_rn(fw[q][0], make_float2(x0, x0), a));
          oo[q] = pack_h2(a.x, a.y);
          if (SPLIT) {
            const float2 lo = __ffma2_rn(unpack_h2(oo[q]), make_float2(-1.0f, -1.0f), a);
            ol[q] = pack_h2(lo.x, lo.y);
          }
        }
      }
      sts128(dst, o);
      if (SPLIT) sts128(dst + Cfg::A_ONE, olo);
    };
    // chunk id (input row u = id / CH) of a tile with any bounds: x samples through xat unless the window is interior
    auto core = [&](int id, bool valid, const uint4& y, const uint4& y2, const uint4& r, const uint4& r2) {
      const int u = id / CH;
      float xm = 0.0f, x0 = 0.0f, xp = 0.0f;
      if (valid) {
        if (PRO == PRO_FIR) {
          if (x_interior) {  // whole window staged: no per-element bounds checks
            const float* xp3 = xraw + (i0 + u - 1 - xs0);
            xm = fin(xp3[0]);
            x0 = fin(xp3[1]);
            xp = fin(xp3[2]);
          } else {
            xm = xat(i0 + u - 1);
            x0 = xat(i0 + u);
            xp = xat(i0 + u + 1);
          }
        } else if (PRO == PRO_NORM_RES_X) {
          x0 = x_interior ? fin(xraw[2 * (i0 + u) - xs0]) : xat(2 * (i0 + u));
        }
      }
      act(valid, xm, x0, xp, y, y2, r, r2, adst + soff_of(u));
    };
    // Hand-over: every transform thread publishes its shared-memory writes to the async proxy, then arrives
    auto hand_over = [&]() {
      fence_proxy_async_smem();
      named_arrive(1 + as, kNamedCount);
      if (!Cfg::DIRECT) named_arrive(1 + NA + rs, kNamedCount);
      if (!Cfg::DIRECT && ++rs == NR) {
        rs = 0;
        rph ^= 1;
      }
      if (++as == NA) {
        as = 0;
        aph ^= 1;
      }
    };
    if constexpr (Cfg::DIRECT) {
      constexpr int NCHUNK = R * CH, NIT = Cfg::NIT, PF = Cfg::PF;
      constexpr int NITP = (NIT + PF - 1) / PF * PF;
      constexpr bool RES = PRO == PRO_NORM_RES;
      struct TileRef {
        const uint8_t* y;  // row i0 of the sample (may lie one row before its start: never dereferenced there)
        const uint8_t* r;
        int i0;
        bool interior;
      };
      auto tile_ref = [&](const TilePos& t, int b) {
        const int ti0 = t.r * POS * STRIDE - 1;
        const long long off = ((long long)b * p.L_in + ti0) * (CIN * 2);
        TileRef tr;
        tr.y = reinterpret_cast<const uint8_t*>(p.in) + off;
        tr.r = RES ? reinterpret_cast<const uint8_t*>(p.in_res) + off : nullptr;
        tr.i0 = ti0;
        tr.interior = (ti0 >= 0) && (ti0 + R <= p.L_in);
        return tr;
      };
      auto chunk_ok = [&](const TileRef& tr, int k, int id) {
        bool ok = (k < NIT - 1) || id < NCHUNK;
        if (!tr.interior) {
          const int i = tr.i0 + id / CH;
          ok = ok && i >= 0 && i < p.L_in;
        }
        return ok;
      };
      auto fetch = [&](const TileRef& tr, int k, uint4& y, uint4& r) {
        const int id = tt + k * NTT;
        if (chunk_ok(tr, k, id)) {
          y = ldg128_stream(tr.y + (size_t)id * 16);
          if (RES) r = ldg128_stream(tr.r + (size_t)id * 16);
        }
      };
      // next tile of this CTA whose sample is live (b < 0: none)
      auto seek = [&](TilePos& t, int& tl) -> int {
        for (; tl < tile_end; ++tl, advance(t)) {
          int bb;
          if (sample_of(t, bb)) return bb;
        }
        return -1;
      };
      const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
      uint4 ybuf[PF], rbuf[PF];
#pragma unroll
      for (int k = 0; k < PF; ++k) ybuf[k] = rbuf[k] = zero4;
      TilePos tp = pos0;
      int tile = tile_begin;
      int b = seek(tp, tile);
      TileRef cur = {nullptr, nullptr, 0, true};
      if (b >= 0) {
        cur = tile_ref(tp, b);
#pragma unroll
        for (int k = 0; k < PF; ++k) fetch(cur, k, ybuf[k], rbuf[k]);
      }
      while (b >= 0) {
        if (b != cur_b) {
          cur_b = b;
          load_consts(b);
        }
        TilePos tn = tp;
        int tilen = tile + 1;
        advance(tn);
        const int bn = seek(tn, tilen);
        TileRef nxt = {nullptr, nullptr, 0, true};
        if (bn >= 0) nxt = tile_ref(tn, bn);
        i0 = cur.i0;
        wc_a.wait(p, &a_empty[as], aph ^ 1);
        adst = smem_u32(sA + as * Cfg::A_BYTES) + (uint32_t)cch * RP * 16;
#pragma unroll
        for (int k = 0; k < NITP; ++k) {
          const int id = tt + k * NTT;
          const uint4 y = ybuf[k % PF], r = rbuf[k % PF];
          // refill the slot: PF chunks ahead, in this tile or (slots of the tail) in the next one
          if (k + PF < NITP) {
            if (k + PF < NIT) fetch(cur, k + PF, ybuf[k % PF], rbuf[k % PF]);
          } else if (k + PF - NITP < NIT) {
            if (bn >= 0) fetch(nxt, k + PF - NITP, ybuf[k % PF], rbuf[k % PF]);
          }
          if (k < NIT && ((k < NIT - 1) || id < NCHUNK)) core(id, chunk_ok(cur, k, id), y, zero4, r, zero4);
        }
        hand_over();
        tp = tn;
        tile = tilen;
        b = bn;
        cur = nxt;
      }
    } else {
    // Interior tiles: chunk k of this thread is chunk tt + k * NTT of the tile, input row u0 + k * UK.  Its raw-stage,
    // x-window and A-stage offsets are the stage base + a per-thread constant (computed once here) + a compile-time
    // constant, the loop over k is fully unrolled and only the last chunk is conditional (on the thread, not the tile).
    constexpr int NK = (R * CH + NTT - 1) / NTT;  // chunks per thread and tile (the last one for some threads only)
    constexpr int UK = NTT / CH;
    static_assert(NTT % CH == 0 && UK % STRIDE == 0, "fixed row stride phase of a thread's chunks");
    const int u0 = tt / CH;
    const bool last_chunk = tt + (NK - 1) * NTT < R * CH;
    const uint32_t raw_t = (uint32_t)tt * (8 * ESZ);
    const uint32_t a_t = soff_of(u0);
    constexpr int XK = (PRO == PRO_NORM_RES_X ? 2 : 1) * UK;  // x-window step between a thread's chunks
    const int x_t = (PRO == PRO_NORM_RES_X ? 2 : 1) * u0;
    TilePos tp = pos0;
    for (int tile = tile_begin; tile < tile_end; ++tile, advance(tp)) {
      int b;
      if (!sample_of(tp, b)) continue;
      if (b != cur_b) {
        cur_b = b;
        load_consts(b);
      }
      const int o0 = tp.r * POS;
      i0 = o0 * STRIDE - 1;
      if (tt == 0 && tile == tile_begin) dbg_ts(p, 3);
      wc_raw.wait(p, &raw_full[rs], rph);
      wc_a.wait(p, &a_empty[as], aph ^ 1);
      if (tt == 0 && tile == tile_begin) dbg_ts(p, 4);
      const uint32_t raw = smem_u32(sRaw + rs * Cfg::RAW_BYTES);
      adst = smem_u32(sA + as * Cfg::A_BYTES) + (uint32_t)cch * RP * 16;
      const bool interior = (i0 >= 0) && (i0 + R <= p.L_in);  // no zero-padding rows in this tile
      xs0 = (PRO == PRO_FIR) ? ((i0 - 1) & ~3) : ((2 * i0) & ~3);
      xraw = reinterpret_cast<const float*>(sRaw + rs * Cfg::RAW_BYTES + Cfg::RAW_ONE);
      x_interior = xs0 >= 0 && xs0 + Cfg::XN <= p.T_raw;
      auto chunk = [&](int id, bool valid) {
        // 8 channels of one input row: one 16-B load (fp16) or two (wide fp32 storage)
        uint4 y = make_uint4(0u, 0u, 0u, 0u), y2 = y, r = y, r2 = y;
        if (valid) {
          if (PRO != PRO_FIR) {
            y = lds128(raw + (uint32_t)id * (8 * ESZ));
            if (WIN) y2 = lds128(raw + (uint32_t)id * 32 + 16);
          }
          if (PRO == PRO_NORM_RES) {
            r = lds128(raw + Cfg::RAW_ONE + (uint32_t)id * (8 * ESZ));
            if (WIN) r2 = lds128(raw + Cfg::RAW_ONE + (uint32_t)id * 32 + 16);
          }
        }
        core(id, valid, y, y2, r, r2);
      };
      // chunk k of an interior tile; xq: this thread's first row in the x window (block-0 fusion modes)
      const uint32_t raw_q = raw + raw_t, a_q = adst + a_t;
      const float* xq = xraw + ((PRO == PRO_FIR ? i0 - 1 : 2 * i0) - xs0 + x_t);
      auto interior_chunk = [&](int k) {
        const uint32_t src = raw_q + (uint32_t)(k * NTT * 8 * ESZ);
        uint4 y = make_uint4(0u, 0u, 0u, 0u), y2 = y, r = y, r2 = y;
        if (PRO != PRO_FIR) {
          y = lds128(src);
          if (WIN) y2 = lds128(src + 16);
        }
        if (PRO == PRO_NORM_RES) {
          r = lds128(src + Cfg::RAW_ONE);
          if (WIN) r2 = lds128(src + Cfg::RAW_ONE + 16);
        }
        float xm = 0.0f, x0 = 0.0f, xp = 0.0f;
        if (PRO == PRO_FIR) {
          xm = fin(xq[k * XK]);
          x0 = fin(xq[k * XK + 1]);
          xp = fin(xq[k * XK + 2]);
        } else if (PRO == PRO_NORM_RES_X) {
          x0 = fin(xq[k * XK]);
        }
        act(true, xm, x0, xp, y, y2, r, r2, a_q + (uint32_t)(k * (UK / STRIDE) * 16));
      };
      if (W2S_DBG(p, 32)) {
      } else if (interior && (Cfg::XN == 0 || x_interior)) {
#pragma unroll
        for (int k = 0; k < NK; ++k) {
          if (k < NK - 1 || last_chunk) interior_chunk(k);
        }
      } else {
        for (int id = tt; id < R * CH; id += NTT) {
          const int i = i0 + id / CH;
          chunk(id, i >= 0 && i < p.L_in);
        }
      }
      hand_over();
    }
    }
    if (tt == 0) {
      wc_a.publish(p, 14);
      if (W2S_DBG(p, 64) && blockIdx.x == 0) g_stream_ts[10] = (unsigned long long)wc_raw.acc;
    }
  }

  // ---------------- teardown ----------------
  tc_fence_before_sync();
  __syncthreads();
  if (tid == 0) dbg_ts(p, 9);
  if (warp == 0) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  if (W2S_DBG(p, 64) && tid == 0 && blockIdx.x < 512) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_stream_cta_ts[2 * blockIdx.x + 1] = t;
  }
}

// SPLIT defaults to the (CIN, COUT) rule of ConvSplit; the wide-storage 64-channel kernels of deep encoders override it.
template <int CIN, int COUT, int STRIDE, int PRO, bool HAS_DS, int MT, int NR, int NA, int NTW, bool WIN = false, bool WOUT = false,
          bool SPLIT = ConvSplit<CIN, COUT>::value>
inline cudaError_t launch_conv_stream(const ConvArgs& a, const ConvArgs* a2, int B, int sm_count, cudaStream_t stream) {
  using Cfg = StreamCfg<CIN, COUT, STRIDE, PRO, HAS_DS, SPLIT, MT, NR, NA, NTW, WIN, WOUT>;
  auto kern = conv_stream_kernel<CIN, COUT, STRIDE, PRO, HAS_DS, SPLIT, MT, NR, NA, NTW, WIN, WOUT>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  const int tiles_per_sample = (a.L_out + Cfg::POS - 1) / Cfg::POS;
  const long long total = (long long)tiles_per_sample * B;
  if (total > 0x7fffffffLL) return cudaErrorInvalidValue;
  const int ctas = sm_count * (Cfg::THREADS <= 384 ? 2 : 1);  // small CTAs run two per SM
  int grid = total < ctas ? (int)total : ctas;
  if (a2 != nullptr && !stream_pairable(COUT, HAS_DS)) return cudaErrorInvalidValue;  // (conv_dispatch never asks for it)
  if (a2 != nullptr) {  // paired launch: half of the grid per group (same B, L for both)
    const int per = total < ctas / 2 ? (int)total : ctas / 2;
    grid = 2 * per;
  }
  const ConvGroup2 g2 = conv_group2(a2);
  kern<<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(a, g2, tiles_per_sample, (int)total);
  return cudaGetLastError();
}

}  // namespace w2s
