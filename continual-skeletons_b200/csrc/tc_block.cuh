// One kernel per block step for the 64-channel CoST-GCN blocks (CoSpatioTemporalBlock, models/base.py:390-446):
//
//   g_n   = relu(BN(sum_i W_i (x_n A_i)) + x_n)                      GraphConvolution        models/base.py:260-270
//   out_n = relu(BN(sum_k Wt_k g_{n-8+k}) + x_{n-4})                 CoTemporalConvolution   :307-334 + delayed residual :417-438
//
// The temporal conv of a 64-channel block is bound by HBM (eight history frames in, one frame out) and leaves the
// tensor pipe ~60 % and the CUDA cores almost entirely idle; the graph conv is bound by CUDA-core work on data that
// is already on chip.  Tiles hold whole skeletons, so both halves of a block step are tile local, and this kernel
// runs them as one software pipeline per token tile:
//
//   TMA: x_n tile (own 32 KB stage) | history ring (4 x 32 KB): g_{n-8} .. g_{n-1}, x_{n-4} | weight ring (3 x 16 KB slabs);
//        three independent producer threads, so a full weight ring never holds up the history stream
//   mix warps      x_n tile -> adjacency-mixed rows X'_i, re-split, tcgen05.st -> TMEM A slots
//   MMA thread     G = [X'_0|X'_1|X'_2|x] [W_0|W_1|W_2|I]^T   (A from TMEM)                      -> TMEM accumulator G
//   epilogue warps G -> +bias, ReLU, split -> ring slot n (the only state write of the graph conv)
//                                             and -> TMEM "newest tap" slot (bf16 hi | lo, K-major)
//   MMA thread     T = sum_{k<8} g_{n-8+k} Wt_k^T + x_{n-4} I^T   (A from the TMA ring)
//                    + g_n Wt_8^T                                  (A from the TMEM tap slot)    -> TMEM accumulator T
//   epilogue warps T -> +bias, ReLU, split -> block-output ring
//
// so g_n is consumed by the temporal conv without a round trip through memory, the graph conv's input tile is the
// same TMA stream as the history frames, and all CUDA-core work of the graph conv runs under the history stream of
// the same or the next tile.  Per tile 12 frames cross HBM (x_n, 8 history, x_{n-4} in; g_n, out_n out) instead of
// 13 for the two separate kernels, in one launch instead of two.
//
// Before the temporal conv's first emission (n < 8 - p) the kernel runs with with_tcn = 0: graph conv only.
//
// TMEM (512 columns): [T accumulator 128 | G accumulator 128 | newest-tap slot 64 | 3 mix slots x 64]; both accumulators
// hold the stacked split-precision form (columns [0,64) hi*hi + lo*hi, [64,128) hi*lo + lo*lo).
// Warps: 0 history producer, 1 MMA issuer + TMEM owner, 2 input-tile producer, 3 weight producer, 4-7 epilogue (G then T
// of every tile), 8-15 mix.
//
// The mix (8 warps, thread = token row = TMEM lane, half of the 64 channels each) works in two passes so that every input
// element is unpacked once instead of once per adjacency entry: (1) the raw hi / lo words of the own row go to registers and,
// unchanged, into the first mix slot (the "plain x" part that carries the identity gcn_residual -- and W_0 when every self
// link is exactly 1); (2) x = hi + lo is written back IN PLACE over the tile as fp32 rows, from which the partitions
// gather with one FMA per adjacency entry and element.
#pragma once
#include "tc_kernels.cuh"

namespace cosk {

constexpr int kPartSrcMax = 4;  // most sources of one output vertex inside partition 1 or 2

enum : unsigned int {
  kDbgMixXFull = 0x08000000u,
  kDbgMixAEmpty = 0x09000000u,
  kDbgMmaAFull = 0x0a000000u,
  kDbgBlkGFull = 0x0b000000u,
  kDbgBlkTapEmpty = 0x0c000000u,
  kDbgBlkTapFull = 0x0d000000u,
  kDbgBlkGEmpty = 0x0e000000u,
};

struct TcBlockArgs {
  CUtensorMap tm_x;     // block input ring (the previous block's output ring) [kOutSlots*2*t_alloc rows][64], box {64, 128}
  CUtensorMap tm_ring;  // this block's temporal ring [kRingSlots*2*t_alloc rows][64], box {64, 128}
  CUtensorMap tm_gw;    // graph-conv weights [128 rows: hi, lo][n_parts*64], box {64, 128}; K-blocks in mix-slot order:
                        // plain x (identity residual [+ W_0 if unit_diag]), [W_0 on a0*x], W_1, W_2
  CUtensorMap tm_tw;    // temporal-conv weights [128 rows: hi, lo][10*64], box {64, 128}; K-block = tap (8 = newest), 9 = identity residual
  int x_row;            // hi-plane row of the input slot (x_n) in tm_x
  int res_row;          // hi-plane row of the delayed input slot (x_{n-4}) in tm_x
  int tap_row[kTaps - 1];  // hi-plane rows of the eight history slots g_{n-8} .. g_{n-1} in tm_ring
  int t_alloc;
  int with_tcn;  // 0: the temporal conv does not emit on this step (graph conv only)
  int n_parts;   // 3: self links are exactly 1 (W_0 folded into the plain-x part); 4: separate a0*x part
  int V;
  int n_tiles, tile_tokens;
  long long n_tokens;
  const int *mix_ptr;
  const int *mix_src;
  const float *mix_val;
  const float *gbias;            // [64] graph conv (BN folded)
  __nv_bfloat16 *g_hi, *g_lo;    // ring slot n (written)
  int cs_g;
  EpiArgs tepi;                  // temporal conv: bias, output slot
  unsigned long long *trace;     // optional phase timers of CTA 0: [32..37] mix {wait x, pass 1+2, gather, wait slot, total, tiles},
                                 // [40..46] MMA {wait G acc, wait mix slot, wait weights, wait T acc, wait history, wait tap, total},
                                 // [48..51] epilogue {wait G, G work, wait T, T work}, [52..55] producers {history wait, weights wait, x wait}
  unsigned int *dbg;
  // (No time-batched form: frame n's temporal conv reads the graph-conv outputs of frames n-8 .. n-1, which a launch covering
  // several frames would be producing concurrently.  cosk_steps with a time chunk runs these blocks as two launches.)
};

struct TcBlockCfg {
  static constexpr int kC = 64;
#ifndef COSK_BLK_HSTAGES
#define COSK_BLK_HSTAGES 4
#define COSK_BLK_BSTAGES 3
#endif
  static constexpr int kHStages = COSK_BLK_HSTAGES;  // history ring
  static constexpr int kBStages = COSK_BLK_BSTAGES;
  static constexpr int kSlabBytes = 2 * kC * kBK * 2;  // 16 KB: [64 hi rows; 64 lo rows] x 64 K
  static constexpr int kXOff = 0;                      // x_n tile: hi plane, lo plane; later the fp32 rows of the same tile
  static constexpr int kHOff = 2 * kABytes;
  static constexpr int kBOff = kHOff + kHStages * 2 * kABytes;
  static constexpr int kBarOff = kBOff + kBStages * kSlabBytes;
  static constexpr int kBiasOff = kBarOff + 512;
  static constexpr int kSmemBytes = kBiasOff + 2 * kC * 4 + 1024;
  static constexpr int kMixSlots = 3;
  static constexpr int kTAcc = 0, kGAcc = 128, kTap = 256, kMix = 320;  // TMEM column offsets
  static constexpr int kTmemCols = 512;
  static_assert(kMix + kMixSlots * 64 <= 512, "TMEM columns");
  static_assert(kSmemBytes <= kSmemLimit, "shared memory budget");
};

// 8 fp32 values -> 4 packed hi words + 4 packed lo words (even channel in the low half, as in memory)
__device__ __forceinline__ void split8(const float (&v)[8], uint32_t *hi, uint32_t *lo) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint32_t h = pack_bf16x2(v[2 * j], v[2 * j + 1]);
    hi[j] = h;
    lo[j] = pack_bf16x2(v[2 * j] - bf16_lo_as_float(h), v[2 * j + 1] - bf16_hi_as_float(h));
  }
}

// byte offset of the 16-byte chunk `c` of row `r` inside a TMA SWIZZLE_128B tile with 128-byte rows
__device__ __forceinline__ uint32_t sw128_off(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }

__global__ void __launch_bounds__(512, 1) k_tc_block64(const __grid_constant__ TcBlockArgs a) {
  using Cfg = TcBlockCfg;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *hfull = reinterpret_cast<uint64_t *>(smem + Cfg::kBarOff);
  uint64_t *hempty = hfull + Cfg::kHStages;
  uint64_t *bfull = hempty + Cfg::kHStages;
  uint64_t *bempty = bfull + Cfg::kBStages;
  uint64_t *mfull = bempty + Cfg::kBStages;
  uint64_t *mempty = mfull + Cfg::kMixSlots;
  uint64_t *xfull = mempty + Cfg::kMixSlots;
  uint64_t *xempty = xfull + 1;
  uint64_t *gfull = xempty + 1;
  uint64_t *gempty = gfull + 1;
  uint64_t *tapfull = gempty + 1;
  uint64_t *tapempty = tapfull + 1;
  uint64_t *tfull = tapempty + 1;
  uint64_t *tempty = tfull + 1;
  uint64_t *mixbar = tempty + 1;  // two rendezvous points of the eight mix warps per tile (mbarriers: bounded waits, unlike bar.sync)
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(mixbar + 2);
  float *gbias_s = reinterpret_cast<float *>(smem + Cfg::kBiasOff);
  float *tbias_s = gbias_s + Cfg::kC;
  const uint32_t smem_base = ptx::smem_u32(smem);
  const int cta = (int)blockIdx.x, ncta = (int)gridDim.x;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kHStages; ++s) {
      ptx::mbar_init(&hfull[s], 1);
      ptx::mbar_init(&hempty[s], 1);
    }
    for (int s = 0; s < Cfg::kBStages; ++s) {
      ptx::mbar_init(&bfull[s], 1);
      ptx::mbar_init(&bempty[s], 1);
    }
    for (int s = 0; s < Cfg::kMixSlots; ++s) {
      ptx::mbar_init(&mfull[s], 8);  // the eight mix warps
      ptx::mbar_init(&mempty[s], 1);
    }
    ptx::mbar_init(xfull, 1);
    ptx::mbar_init(xempty, 8);
    ptx::mbar_init(gfull, 1);
    ptx::mbar_init(gempty, 4);  // the four epilogue warps
    ptx::mbar_init(tapfull, 4);
    ptx::mbar_init(tapempty, 1);
    ptx::mbar_init(tfull, 1);
    ptx::mbar_init(tempty, 4);
    ptx::mbar_init(&mixbar[0], 8);
    ptx::mbar_init(&mixbar[1], 8);
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&a.tm_x);
    ptx::prefetch_tmap(&a.tm_ring);
    ptx::prefetch_tmap(&a.tm_gw);
    ptx::prefetch_tmap(&a.tm_tw);
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish();
  }
  for (int i = threadIdx.x; i < Cfg::kC; i += blockDim.x) {
    gbias_s[i] = a.gbias[i];
    tbias_s[i] = a.tepi.bias[i];
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();  // prologue above touched only static data; activations of the previous kernel from here on
  const bool with_tcn = a.with_tcn != 0;
  const int P = a.n_parts;
  const int n_items = a.n_tiles;
  const bool tr0 = a.trace != nullptr && cta == 0;

  if (warp == 0) {
    // ---- history producer: g_{n-8} .. g_{n-1} and x_{n-4} of every tile, in the order the temporal GEMM eats them ----
    if (lane == 0 && with_tcn) {
      PipeState ph;
      bool ok = true;
      unsigned long long tw = 0;
      for (int tile = cta; ok && tile < n_items; tile += ncta) {
        const int tok0 = tile * a.tile_tokens;
        for (int k = 0; k < kTaps; ++k) {
          const long long w0 = tr0 ? clock64() : 0;
          ok = ptx::mbar_wait(&hempty[ph.stage], ph.phase ^ 1, a.dbg, kDbgProdEmpty | (unsigned)k);
          if (!ok) break;
          if (tr0) tw += clock64() - w0;
          const uint32_t sa = smem_base + Cfg::kHOff + ph.stage * 2 * kABytes;
          const CUtensorMap *tm = k < kTaps - 1 ? &a.tm_ring : &a.tm_x;
          const int row = (k < kTaps - 1 ? a.tap_row[k] : a.res_row) + tok0;
          ptx::mbar_arrive_expect_tx(&hfull[ph.stage], 2 * kABytes);
          ptx::tma_load_2d_hint(sa, tm, &hfull[ph.stage], 0, row, ptx::kEvictFirst);
          ptx::tma_load_2d_hint(sa + kABytes, tm, &hfull[ph.stage], 0, row + a.t_alloc, ptx::kEvictFirst);
          ph.advance<Cfg::kHStages>();
        }
      }
      if (tr0) a.trace[52] = tw;
    }
  } else if (warp == 2) {
    // ---- input-tile producer: x_n of the next tile as soon as the mix warps are done with the current one ----------
    if (lane == 0) {
      bool ok = true;
      int it = 0;
      unsigned long long tw = 0;
      for (int tile = cta; ok && tile < n_items; tile += ncta, ++it) {
        const long long w0 = tr0 ? clock64() : 0;
        ok = ptx::mbar_wait(xempty, (uint32_t)((it & 1) ^ 1), a.dbg, kDbgProdEmpty | 0x400000u | (unsigned)it);
        if (!ok) break;
        if (tr0) tw += clock64() - w0;
        const int row = a.x_row + tile * a.tile_tokens;
        ptx::mbar_arrive_expect_tx(xfull, 2 * kABytes);
        // x_n is read again four steps from now (as the delayed residual) but not before: no reason to keep it in L2
        ptx::tma_load_2d_hint(smem_base + Cfg::kXOff, &a.tm_x, xfull, 0, row, ptx::kEvictFirst);
        ptx::tma_load_2d_hint(smem_base + Cfg::kXOff + kABytes, &a.tm_x, xfull, 0, row + a.t_alloc, ptx::kEvictFirst);
      }
      if (tr0) a.trace[54] = tw;
    }
  } else if (warp == 3) {
    // ---- weight producer: graph-conv slabs, then the temporal taps in GEMM order (residual before the newest tap) ----
    if (lane == 0) {
      PipeState pb;
      bool ok = true;
      unsigned long long tw = 0;
      auto load_b = [&](const CUtensorMap *tm, int kb) {
        const long long w0 = tr0 ? clock64() : 0;
        ok = ptx::mbar_wait(&bempty[pb.stage], pb.phase ^ 1, a.dbg, kDbgProdEmpty | 0x800000u | (unsigned)kb);
        if (!ok) return;
        if (tr0) tw += clock64() - w0;
        const uint32_t sb = smem_base + Cfg::kBOff + pb.stage * Cfg::kSlabBytes;
        ptx::mbar_arrive_expect_tx(&bfull[pb.stage], Cfg::kSlabBytes);
        ptx::tma_load_2d_hint(sb, tm, &bfull[pb.stage], kb * kBK, 0, ptx::kEvictLast);
        pb.advance<Cfg::kBStages>();
      };
      for (int tile = cta; ok && tile < n_items; tile += ncta) {
        for (int p = 0; ok && p < P; ++p) load_b(&a.tm_gw, p);
        if (with_tcn) {
          for (int k = 0; ok && k < kTaps - 1; ++k) load_b(&a.tm_tw, k);
          if (ok) load_b(&a.tm_tw, kTaps);      // identity weights of the delayed residual
          if (ok) load_b(&a.tm_tw, kTaps - 1);  // newest tap (its A operand comes from TMEM)
        }
      }
      if (tr0) a.trace[53] = tw;
    }
  } else if (warp == 1) {
    if (lane == 0) {
      PipeState ph, pb, pm;
      bool ok = true;
      int it = 0;
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(kTileRows, 2 * Cfg::kC);
      unsigned long long tw[6] = {0, 0, 0, 0, 0, 0};
      const long long tstart = tr0 ? clock64() : 0;
      long long w0 = 0;
      auto lap = [&](int i) {
        if (tr0) {
          const long long n_ = clock64();
          tw[i] += n_ - w0;
          w0 = n_;
        }
      };
      for (int tile = cta; ok && tile < n_items; tile += ncta, ++it) {
        const uint32_t par = (uint32_t)(it & 1);
        // ---- graph conv: G = sum_p X'_p W_p^T, A operand in the mix slots -------------------------------
        if (tr0) w0 = clock64();
        ok = ptx::mbar_wait(gempty, par ^ 1, a.dbg, kDbgBlkGEmpty | (unsigned)it);
        if (!ok) break;
        lap(0);
        ptx::tc_fence_after();
        for (int p = 0; p < P; ++p) {
          ok = ptx::mbar_wait(&mfull[pm.stage], pm.phase, a.dbg, kDbgMmaAFull | (unsigned)p);
          if (!ok) break;
          lap(1);
          ok = ptx::mbar_wait(&bfull[pb.stage], pb.phase, a.dbg, kDbgMmaFull | 0x400000u | (unsigned)p);
          if (!ok) break;
          lap(2);
          ptx::tc_fence_after();
          const uint32_t ta = tmem_base + Cfg::kMix + pm.stage * 64;
          const uint32_t bs = ptx::umma_desc_lo(smem_base + Cfg::kBOff + pb.stage * Cfg::kSlabBytes);
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k) {
            ptx::umma_bf16_ts(tmem_base + Cfg::kGAcc, ta + 8 * k, bs + 2 * k, idesc, (p == 0 && k == 0) ? 0u : 1u);
            ptx::umma_bf16_ts(tmem_base + Cfg::kGAcc, ta + 32 + 8 * k, bs + 2 * k, idesc, 1u);
          }
          ptx::umma_commit(&mempty[pm.stage]);
          ptx::umma_commit(&bempty[pb.stage]);
          pm.advance<Cfg::kMixSlots>();
          pb.advance<Cfg::kBStages>();
        }
        if (!ok) break;
        ptx::umma_commit(gfull);
        if (!with_tcn) continue;
        // ---- temporal conv: eight history frames and the delayed input from the TMA ring ... --------------
        if (tr0) w0 = clock64();
        ok = ptx::mbar_wait(tempty, par ^ 1, a.dbg, kDbgMmaTmemEmpty | (unsigned)it);
        if (!ok) break;
        lap(3);
        ptx::tc_fence_after();
        for (int kb = 0; kb < kTaps; ++kb) {
          ok = ptx::mbar_wait(&hfull[ph.stage], ph.phase, a.dbg, kDbgMmaFull | (unsigned)kb);
          if (!ok) break;
          ok = ptx::mbar_wait(&bfull[pb.stage], pb.phase, a.dbg, kDbgMmaFull | 0x800000u | (unsigned)kb);
          if (!ok) break;
          lap(4);
          ptx::tc_fence_after();
          const uint32_t sa = smem_base + Cfg::kHOff + ph.stage * 2 * kABytes;
          const uint32_t sb = smem_base + Cfg::kBOff + pb.stage * Cfg::kSlabBytes;
          issue_kblock_stacked<2 * Cfg::kC>(tmem_base + Cfg::kTAcc, sa, sa + kABytes, sb, kb == 0);
          ptx::umma_commit(&hempty[ph.stage]);
          ptx::umma_commit(&bempty[pb.stage]);
          ph.advance<Cfg::kHStages>();
          pb.advance<Cfg::kBStages>();
        }
        if (!ok) break;
        // ---- ... and the newest frame g_n straight from tensor memory ------------------------------------
        ok = ptx::mbar_wait(tapfull, par, a.dbg, kDbgBlkTapFull | (unsigned)it);
        if (!ok) break;
        ok = ptx::mbar_wait(&bfull[pb.stage], pb.phase, a.dbg, kDbgMmaFull | 0xc00000u);
        if (!ok) break;
        lap(5);
        ptx::tc_fence_after();
        {
          const uint32_t ta = tmem_base + Cfg::kTap;
          const uint32_t bs = ptx::umma_desc_lo(smem_base + Cfg::kBOff + pb.stage * Cfg::kSlabBytes);
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k) {
            ptx::umma_bf16_ts(tmem_base + Cfg::kTAcc, ta + 8 * k, bs + 2 * k, idesc, 1u);
            ptx::umma_bf16_ts(tmem_base + Cfg::kTAcc, ta + 32 + 8 * k, bs + 2 * k, idesc, 1u);
          }
          ptx::umma_commit(tapempty);
          ptx::umma_commit(&bempty[pb.stage]);
          pb.advance<Cfg::kBStages>();
        }
        ptx::umma_commit(tfull);
      }
      if (tr0) {
        for (int i = 0; i < 6; ++i) a.trace[40 + i] = tw[i];
        a.trace[46] = clock64() - tstart;
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ---- epilogue: G of the tile (ring write + newest-tap operand), then T of the tile ---------------------
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
    bool ok = true;
    int it = 0;
    const bool tr = tr0 && q == 0 && lane == 0;
    unsigned long long tw[4] = {0, 0, 0, 0};
    long long w0 = 0;
    auto lap = [&](int i) {
      if (tr) {
        const long long n_ = clock64();
        tw[i] += n_ - w0;
        w0 = n_;
      }
    };
    for (int tile = cta; ok && tile < n_items; tile += ncta, ++it) {
      const uint32_t par = (uint32_t)(it & 1);
      const long long tok = (long long)tile * a.tile_tokens + row;
      const bool valid = row < a.tile_tokens && tok < a.n_tokens;
      if (tr) w0 = clock64();
      ok = ptx::mbar_wait(gfull, par, a.dbg, kDbgBlkGFull | (unsigned)it);
      if (!ok) break;
      lap(0);
      ptx::tc_fence_after();
#pragma unroll 1
      for (int half = 0; half < 2; ++half) {
        const int c0 = 32 * half;
        uint32_t r[32];
        float v[32];
        ptx::tmem_ld_32x32(lane_base + Cfg::kGAcc + c0, r);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        ptx::tmem_ld_32x32(lane_base + Cfg::kGAcc + Cfg::kC + c0, r);
        ptx::tmem_ld_wait();
        uint32_t oh[16], ol[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float x0 = fmaxf(v[2 * j] + __uint_as_float(r[2 * j]) + gbias_s[c0 + 2 * j], 0.f);
          const float x1 = fmaxf(v[2 * j + 1] + __uint_as_float(r[2 * j + 1]) + gbias_s[c0 + 2 * j + 1], 0.f);
          const uint32_t h = pack_bf16x2(x0, x1);
          oh[j] = h;
          ol[j] = pack_bf16x2(x0 - bf16_lo_as_float(h), x1 - bf16_hi_as_float(h));
        }
        if (valid) {
          uint4 *qh = reinterpret_cast<uint4 *>(a.g_hi + tok * a.cs_g + c0);
          uint4 *ql = reinterpret_cast<uint4 *>(a.g_lo + tok * a.cs_g + c0);
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            ptx::stg_v4(qh + w, make_uint4(oh[4 * w], oh[4 * w + 1], oh[4 * w + 2], oh[4 * w + 3]));
            ptx::stg_v4(ql + w, make_uint4(ol[4 * w], ol[4 * w + 1], ol[4 * w + 2], ol[4 * w + 3]));
          }
        }
        if (with_tcn) {
          if (half == 0) {  // the temporal conv of the previous tile is done reading the tap slot
            ok = ptx::mbar_wait(tapempty, par ^ 1, a.dbg, kDbgBlkTapEmpty | (unsigned)it);
            if (!ok) break;
            ptx::tc_fence_after();
          }
          // K-major bf16 operand row: channels (2j, 2j+1) of this chunk in column 16*half + j, hi plane then lo plane
          ptx::tmem_st_32x16(lane_base + Cfg::kTap + 16 * half, oh);
          ptx::tmem_st_32x16(lane_base + Cfg::kTap + 32 + 16 * half, ol);
        }
      }
      if (!ok) break;
      if (with_tcn) ptx::tmem_st_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive(gempty);  // G accumulator drained: the next tile's graph conv may overwrite it
        if (with_tcn) ptx::mbar_arrive(tapfull);
      }
      lap(1);
      if (!with_tcn) continue;
      ok = ptx::mbar_wait(tfull, par, a.dbg, kDbgEpiTmemFull | (unsigned)it);
      if (!ok) break;
      lap(2);
      ptx::tc_fence_after();
      epilogue_rows<Cfg::kC, true>(lane_base + Cfg::kTAcc, tbias_s, a.tepi, tok, valid);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(tempty);
      lap(3);
    }
    if (tr)
      for (int i = 0; i < 4; ++i) a.trace[48 + i] = tw[i];
  } else if (warp >= 8) {
    // ---- mix: thread = token row (TMEM lane), this warp's half of the 64 channels ------------------------------
    const int q = warp & 3, h = (warp - 8) >> 2;
    const int row = q * 32 + lane;
    // CSR of this row (tile invariant: tiles are skeleton aligned).  Sources as byte offset of the fp32 row + swizzle key;
    // unused entries carry a zero coefficient and point at the own row; loops run to the warp's maximum count.
    uint32_t s_off[2][kPartSrcMax];  // the key is bits 8..10 of the offset
    float s_cf[2][kPartSrcMax];
    int nmax[2] = {0, 0};
    float d0 = 0.f;
    {
      const int wv = row % a.V, sk0 = row - wv;
      const bool live = row < a.tile_tokens;
      if (live) {
        const int e0 = a.mix_ptr[wv];
        if (a.mix_ptr[wv + 1] > e0) d0 = a.mix_val[e0];
      }
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        const int eb = a.mix_ptr[(p + 1) * a.V + wv], ee = a.mix_ptr[(p + 1) * a.V + wv + 1];
        const int n = live ? min(ee - eb, kPartSrcMax) : 0;
#pragma unroll
        for (int e = 0; e < kPartSrcMax; ++e) {
          const bool on = e < n;
          const int sr = on ? sk0 + a.mix_src[eb + e] : row;
          s_off[p][e] = (uint32_t)sr * 256u;
          s_cf[p][e] = on ? a.mix_val[eb + e] : 0.f;
        }
        int m = n;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
        nmax[p] = m;
      }
    }
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + Cfg::kMix + 16 * h;
    uint8_t *xs = smem + Cfg::kXOff;
    PipeState pm;
    bool ok = true;
    int it = 0;
    const bool tr = tr0 && warp == 8 && lane == 0;
    unsigned long long tw[4] = {0, 0, 0, 0};
    long long tc = 0;
    const long long tstart = tr ? clock64() : 0;
    auto lap = [&](int i) {
      if (tr) {
        const long long n_ = clock64();
        tw[i] += n_ - tc;
        tc = n_;
      }
    };
    // one finished part -> its mix slot in tensor memory
    auto put = [&](const uint32_t (&oh)[16], const uint32_t (&ol)[16], unsigned code) {
      lap(code == 0 ? 1 : 2);
      ok = ptx::mbar_wait(&mempty[pm.stage], pm.phase ^ 1, a.dbg, kDbgMixAEmpty | code);
      if (!ok) return;
      lap(3);
      ptx::tc_fence_after();
      const uint32_t ta = lane_addr + pm.stage * 64;
      ptx::tmem_st_32x16(ta, oh);
      ptx::tmem_st_32x16(ta + 32, ol);
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&mfull[pm.stage]);
      pm.advance<Cfg::kMixSlots>();
    };
    // rendezvous of the mix warps: release / acquire through an mbarrier, so a failed pipeline cannot park a warp forever
    auto mix_sync = [&](int which, uint32_t parity) {
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&mixbar[which]);
      ok = ptx::mbar_wait(&mixbar[which], parity, a.dbg, kDbgMixXFull | 0x800000u | (unsigned)which);
    };
    for (int tile = cta; ok && tile < n_items; tile += ncta, ++it) {
      if (tr) tc = clock64();
      ok = ptx::mbar_wait(xfull, (uint32_t)(it & 1), a.dbg, kDbgMixXFull | (unsigned)it);
      if (!ok) break;
      lap(0);
      // pass 1: own row, raw words: 4 chunks of 8 channels per plane
      uint32_t rh[16], rl[16];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t off = sw128_off(row, 4 * h + j);
        const uint4 hv = *reinterpret_cast<const uint4 *>(xs + off);
        const uint4 lv = *reinterpret_cast<const uint4 *>(xs + kABytes + off);
        rh[4 * j] = hv.x; rh[4 * j + 1] = hv.y; rh[4 * j + 2] = hv.z; rh[4 * j + 3] = hv.w;
        rl[4 * j] = lv.x; rl[4 * j + 1] = lv.y; rl[4 * j + 2] = lv.z; rl[4 * j + 3] = lv.w;
      }
      mix_sync(0, (uint32_t)(it & 1));  // every raw word of the tile is in registers: the tile may be overwritten
      if (!ok) break;
      // pass 2: x = hi + lo as fp32, in place: row r at bytes [256 r, 256 r + 256), 16-byte chunks XOR-swizzled with r & 7
#pragma unroll
      for (int b = 0; b < 8; ++b) {
        const float4 f4 = make_float4(bf16_lo_as_float(rh[2 * b]) + bf16_lo_as_float(rl[2 * b]), bf16_hi_as_float(rh[2 * b]) + bf16_hi_as_float(rl[2 * b]),
                                      bf16_lo_as_float(rh[2 * b + 1]) + bf16_lo_as_float(rl[2 * b + 1]),
                                      bf16_hi_as_float(rh[2 * b + 1]) + bf16_hi_as_float(rl[2 * b + 1]));
        *reinterpret_cast<float4 *>(xs + row * 256 + (((8 * h + b) ^ (row & 7)) << 4)) = f4;
      }
      put(rh, rl, 0);  // part "plain x": the words pass through unchanged
      if (!ok) break;
      if (P == 4) {  // self links with a coefficient other than 1: a0 * x from the own registers
        uint32_t oh[16], ol[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float a8[8];
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            a8[2 * w] = d0 * (bf16_lo_as_float(rh[4 * j + w]) + bf16_lo_as_float(rl[4 * j + w]));
            a8[2 * w + 1] = d0 * (bf16_hi_as_float(rh[4 * j + w]) + bf16_hi_as_float(rl[4 * j + w]));
          }
          split8(a8, oh + 4 * j, ol + 4 * j);
        }
        put(oh, ol, 1);
        if (!ok) break;
      }
      mix_sync(1, (uint32_t)(it & 1));  // fp32 tile complete
      if (!ok) break;
#pragma unroll
      for (int pp = 0; pp < 2; ++pp) {
        const int n = nmax[pp];
        uint32_t oh[16], ol[16];
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {  // 16 channels at a time: four 16-byte loads in flight per adjacency entry
          float acc[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) acc[e] = 0.f;
#pragma unroll
          for (int e = 0; e < kPartSrcMax; ++e) {
            if (e < n) {
              const uint32_t off = s_off[pp][e];
              const uint8_t *base = xs + off;
              const uint32_t key = (off >> 8) & 7u;
              float4 v[4];
#pragma unroll
              for (int b = 0; b < 4; ++b) v[b] = *reinterpret_cast<const float4 *>(base + (((uint32_t)(8 * h + 4 * jj + b) ^ key) << 4));
              const float cf = s_cf[pp][e];
#pragma unroll
              for (int b = 0; b < 4; ++b) {
                acc[4 * b] = fmaf(cf, v[b].x, acc[4 * b]);
                acc[4 * b + 1] = fmaf(cf, v[b].y, acc[4 * b + 1]);
                acc[4 * b + 2] = fmaf(cf, v[b].z, acc[4 * b + 2]);
                acc[4 * b + 3] = fmaf(cf, v[b].w, acc[4 * b + 3]);
              }
            }
          }
          float lo8[8], hi8[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            lo8[e] = acc[e];
            hi8[e] = acc[8 + e];
          }
          split8(lo8, oh + 8 * jj, ol + 8 * jj);
          split8(hi8, oh + 8 * jj + 4, ol + 8 * jj + 4);
        }
        put(oh, ol, 2 + pp);
        if (!ok) break;
      }
      if (!ok) break;
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(xempty);  // this warp is done with the tile: the next x_n may land
    }
    if (tr) {
      for (int i = 0; i < 4; ++i) a.trace[32 + i] = tw[i];
      a.trace[36] = clock64() - tstart;
      a.trace[37] = (unsigned long long)it;
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

}  // namespace cosk
