// tcgen05 / TMEM / TMA tile kernels for the two dense contractions of a CoST-GCN block step.
//
// Orientation: D[128 tokens x COUT] += A[128 tokens x 64] * B[COUT x 64]^T per K-block, i.e. the
// token rows of 5 skeletons (125 of 128 rows valid for V = 25) are the UMMA M dimension and the
// BN-folded weights are the N x K operand.  State and weights are split-bf16 (hi/lo planes); every
// K-block issues the three products hi*hi + lo*hi + hi*lo into one fp32 TMEM accumulator.
//
//   k_tc_tcn<COUT>      9-tap temporal conv over the ring (+ folded strided residual conv as extra
//                       K-blocks) + bias + identity residual + ReLU.     A and B arrive by TMA.
//   k_tc_gcn<P>         graph conv as GEMM-then-mix: Y = X [W_0|W_1|W_2(|W_r)]^T on tcgen05 for 64
//                       output channels per pass, then the sparse adjacency row combination of the
//                       fp32 accumulators in the epilogue (through shared memory, CSR in registers);
//                       bias + identity residual + ReLU; result -> ring slot.
//
// Both are persistent (one CTA per SM loops over token tiles) and warp specialised:
//   warp 0  TMA producer     warp 1  MMA issuer + TMEM owner     warps 4-7  epilogue
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace cosk {

constexpr int kBK = 64;                      // K elements per block = one 128-byte swizzle row
constexpr int kABytes = kTileRows * kBK * 2; // 16 KB per plane
constexpr int kSmemLimit = 232448;           // 227 KB opt-in maximum per CTA

// error codes written to the debug word when a bounded wait expires: role << 24 | stage info
enum : unsigned int {
  kDbgProdEmpty = 0x01000000u,
  kDbgMmaFull = 0x02000000u,
  kDbgMmaTmemEmpty = 0x03000000u,
  kDbgEpiTmemFull = 0x04000000u,
  kDbgEpiExchEmpty = 0x05000000u,
  kDbgEpiExchFull = 0x06000000u,
};

struct PipeState {
  int stage = 0;
  uint32_t phase = 0;
  template <int N>
  __device__ __forceinline__ void advance() {
    if (++stage == N) {
      stage = 0;
      phase ^= 1;
    }
  }
};

// The three split-precision products of one K-block (4 UMMA K-steps each).
template <int COUT>
__device__ __forceinline__ void issue_kblock(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                             bool first) {
  constexpr uint32_t idesc = ptx::umma_idesc_bf16(kTileRows, COUT);
  const uint32_t ah = ptx::umma_desc_lo(a_hi), al = ptx::umma_desc_lo(a_lo), bh = ptx::umma_desc_lo(b_hi), bl = ptx::umma_desc_lo(b_lo);
#pragma unroll
  for (int k = 0; k < kBK / 16; ++k) {  // one UMMA K-step = 32 bytes = 2 descriptor units
    ptx::umma_bf16_lo(tmem_d, ah + 2 * k, bh + 2 * k, idesc, (first && k == 0) ? 0u : 1u);
    ptx::umma_bf16_lo(tmem_d, al + 2 * k, bh + 2 * k, idesc, 1u);
    ptx::umma_bf16_lo(tmem_d, ah + 2 * k, bl + 2 * k, idesc, 1u);
  }
}

// "Stacked-B" form of the split-precision product for COUT <= 128: the weight tile's hi and lo planes sit
// back to back in shared memory and are used as ONE operand of N' = 2*COUT rows, so a K-step is two MMAs
// (A_hi and A_lo against [B_hi; B_lo]) instead of three.  Accumulator columns [0, COUT) collect
// hi*hi + lo*hi, columns [COUT, 2*COUT) collect hi*lo + lo*lo; the epilogue adds the two halves.  A
// tcgen05.mma costs a fixed ~85 cycles (the 128-row A fetch) plus ~0.2 cycles per accumulator column, so
// fewer, wider instructions are what makes the narrow layers faster (and the lo*lo term comes for free).
template <int N2>
__device__ __forceinline__ void issue_kblock_stacked(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_stack, bool first) {
  constexpr uint32_t idesc = ptx::umma_idesc_bf16(kTileRows, N2);
  const uint32_t ah = ptx::umma_desc_lo(a_hi), al = ptx::umma_desc_lo(a_lo), bs = ptx::umma_desc_lo(b_stack);
#pragma unroll
  for (int k = 0; k < kBK / 16; ++k) {
    ptx::umma_bf16_lo(tmem_d, ah + 2 * k, bs + 2 * k, idesc, (first && k == 0) ? 0u : 1u);
    ptx::umma_bf16_lo(tmem_d, al + 2 * k, bs + 2 * k, idesc, 1u);
  }
}

struct EpiArgs {
  const float *bias;                // [COUT]
  const __nv_bfloat16 *r_hi, *r_lo; // identity residual rows (nullptr: none)
  int cs_r;
  __nv_bfloat16 *y_hi, *y_lo;
  int cs_out;
  float floor = 0.f;  // lower clamp of the output: 0 = ReLU; -inf when the kernel serves as a plain GEMM (qkv conv)
};

// One epilogue warp: 32 accumulator rows, COUT fp32 columns each -> bias, residual, ReLU, split,
// 128-bit stores of the row's channel vector.
template <int COUT, bool STACKED>
__device__ __forceinline__ void epilogue_rows(uint32_t taddr_row0, const float *bias_s, const EpiArgs &e, long long tok,
                                              bool valid) {
#pragma unroll 1
  for (int c0 = 0; c0 < COUT; c0 += 32) {
    uint32_t r[32];
    ptx::tmem_ld_32x32(taddr_row0 + c0, r);
    ptx::tmem_ld_wait();
    float v[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
    if (STACKED) {  // second half of the stacked accumulator: hi*lo + lo*lo
      ptx::tmem_ld_32x32(taddr_row0 + COUT + c0, r);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] += __uint_as_float(r[j]);
    }
    if (valid) {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] += bias_s[c0 + j];
      if (e.r_hi != nullptr) {
        const uint4 *ph = reinterpret_cast<const uint4 *>(e.r_hi + tok * e.cs_r + c0);
        const uint4 *pl = reinterpret_cast<const uint4 *>(e.r_lo + tok * e.cs_r + c0);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint4 h = ptx::ldg_v4(ph + q), l = ptx::ldg_v4(pl + q);
          const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            v[q * 8 + w * 2] += bf16_lo_as_float(hw[w]) + bf16_lo_as_float(lw[w]);
            v[q * 8 + w * 2 + 1] += bf16_hi_as_float(hw[w]) + bf16_hi_as_float(lw[w]);
          }
        }
      }
      uint32_t oh[16], ol[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float x0 = fmaxf(v[2 * j], e.floor), x1 = fmaxf(v[2 * j + 1], e.floor);
        const uint32_t h = pack_bf16x2(x0, x1);
        oh[j] = h;
        ol[j] = pack_bf16x2(x0 - bf16_lo_as_float(h), x1 - bf16_hi_as_float(h));
      }
      uint4 *qh = reinterpret_cast<uint4 *>(e.y_hi + tok * e.cs_out + c0);
      uint4 *ql = reinterpret_cast<uint4 *>(e.y_lo + tok * e.cs_out + c0);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        ptx::stg_v4(qh + q, make_uint4(oh[4 * q], oh[4 * q + 1], oh[4 * q + 2], oh[4 * q + 3]));
        ptx::stg_v4(ql + q, make_uint4(ol[4 * q], ol[4 * q + 1], ol[4 * q + 2], ol[4 * q + 3]));
      }
    }
  }
}

// =============================================================================================
// temporal conv
// =============================================================================================
struct TcTcnArgs {
  CUtensorMap tm_ring;  // [slots*2*t_alloc rows][C]   box {64, 128}
  CUtensorMap tm_res;   // previous block's output ring [kOutSlots*2*t_alloc rows][Cr], box {64, 128}
  CUtensorMap tm_w;     // [2*COUT rows (hi then lo)][9*C + Cr]  box {64, COUT}
  int tap_row[kTaps];   // first row of the hi plane of each tap's slot (oldest .. newest)
  int res_row;          // first row of the hi plane of the residual slot
  int t_alloc;          // rows per plane
  int n_taps;           // kTaps; 1 when the kernel serves as the output conv of the self-attention unit (operand = tap_row[0])
  int kb_per_tap;       // C / 64
  int kb_res;           // Cr / 64 when res_kind == 2 else 0
  int n_tiles, tile_tokens;
  int reverse;  // 1: every CTA walks its own tiles (c, c + grid, ...) from the last to the first: the graph conv that
                // produced the newest tap walked them first to last on the same CTA index (same SM / L2 partition),
                // so the most recently written rows -- the ones still in L2 -- are consumed first
  long long n_tokens;
  EpiArgs epi;
  unsigned long long *trace;  // optional phase timers of CTA 0 (COSK_TRACE=1): [24] producer wait, [25] producer total,
                              // [26] MMA wait operands, [27] MMA wait accumulator, [28] MMA total
  unsigned int *dbg;
  // time-batched launch (n_frames > 1): frame f reads taps from slots (tap_walk.slot(f) + k) % tap_walk.slots of the temporal
  // ring, the delayed input from res_walk.slot(f) of the input ring, and writes out_walk.slot(f) of the output ring;
  // epi.y_* / epi.r_* then point at slot 0 of their rings.  n_frames == 1: tap_row / res_row / epi as given.
  int n_frames = 1;
  int slot_rows = 0;  // rows per ring slot (2 * t_alloc)
  RingWalk tap_walk, res_walk, out_walk;
  long long out_slot_elems = 0, res_slot_elems = 0;
};

// rows and pointers of frame f of a (possibly time-batched) temporal-conv launch
__device__ __forceinline__ int tcn_tap_row(const TcTcnArgs &a, int f, int tap) {
  return a.n_frames == 1 ? a.tap_row[tap] : ((a.tap_walk.slot(f) + tap) % a.tap_walk.slots) * a.slot_rows;
}
__device__ __forceinline__ int tcn_res_row(const TcTcnArgs &a, int f) {
  return a.n_frames == 1 ? a.res_row : a.res_walk.slot(f) * a.slot_rows;
}
__device__ __forceinline__ EpiArgs tcn_epi(const TcTcnArgs &a, int f) {
  EpiArgs e = a.epi;
  if (a.n_frames > 1) {
    const long long o = (long long)a.out_walk.slot(f) * a.out_slot_elems;
    e.y_hi += o;
    e.y_lo += o;
    if (e.r_hi != nullptr) {
      const long long r = (long long)a.res_walk.slot(f) * a.res_slot_elems;
      e.r_hi += r;
      e.r_lo += r;
    }
  }
  return e;
}

template <int COUT>
struct TcTcnCfg {
  // Activations (HBM latency) and weights (L2 latency) travel in separate rings so that the
  // activation ring can be one stage deeper where shared memory is tight (COUT = 256).
  static constexpr int kBBytes = COUT * kBK * 2;
  static constexpr int kAStages = COUT == 64 ? 5 : 3;
  static constexpr int kBStages = COUT == 64 ? 3 : (COUT == 128 ? 3 : 2);
  static constexpr int kAOff = 0;
  static constexpr int kBOff = kAStages * 2 * kABytes;
  static constexpr int kBarOff = kBOff + kBStages * 2 * kBBytes;
  static constexpr int kBiasOff = kBarOff + 256;
  static constexpr int kSmemBytes = kBiasOff + COUT * 4 + 1024;  // + slack for manual 1024-B alignment
  static constexpr bool kStacked = COUT <= 128;                  // two MMAs per K-step against [B_hi; B_lo]
  static constexpr int kAccCols = kStacked ? 2 * COUT : COUT;
  static constexpr int kTmemCols = 2 * kAccCols;                 // double-buffered accumulator
  static_assert(kSmemBytes <= kSmemLimit, "shared memory budget");
  static_assert(kTmemCols <= 512 && (kTmemCols & (kTmemCols - 1)) == 0, "TMEM columns");
};

template <int COUT>
__device__ __forceinline__ void tcn_body(const TcTcnArgs &a, uint8_t *smem_raw, const int cta, const int ncta) {
  using Cfg = TcTcnCfg<COUT>;
  // SWIZZLE_128B tiles need 1024-byte alignment in the shared window: align on the shared address
  uint8_t *smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *afull = reinterpret_cast<uint64_t *>(smem + Cfg::kBarOff);
  uint64_t *aempty = afull + Cfg::kAStages;
  uint64_t *bfull = aempty + Cfg::kAStages;
  uint64_t *bempty = bfull + Cfg::kBStages;
  uint64_t *tfull = bempty + Cfg::kBStages;
  uint64_t *tempty = tfull + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + 2);
  float *bias_s = reinterpret_cast<float *>(smem + Cfg::kBiasOff);
  const uint32_t smem_base = ptx::smem_u32(smem);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kAStages; ++s) {
      ptx::mbar_init(&afull[s], 1);
      ptx::mbar_init(&aempty[s], 1);
    }
    for (int s = 0; s < Cfg::kBStages; ++s) {
      ptx::mbar_init(&bfull[s], 1);
      ptx::mbar_init(&bempty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], 4);
    }
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&a.tm_ring);
    ptx::prefetch_tmap(&a.tm_w);
    if (a.kb_res) ptx::prefetch_tmap(&a.tm_res);
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish();
  }
  for (int i = threadIdx.x; i < COUT; i += blockDim.x) bias_s[i] = a.epi.bias[i];
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();  // prologue above touched only static data; activations of the previous kernel from here on
  const int nkb = a.n_taps * a.kb_per_tap + a.kb_res;
  const int n_items = a.n_tiles * a.n_frames;  // (frame, tile) work items

  if (warp == 0) {
    if (lane == 0) {
      PipeState pa, pb;
      bool ok = true;
      const bool tr = a.trace != nullptr && cta == 0;
      unsigned long long tw = 0;
      const long long tstart = tr ? clock64() : 0;
      for (int ti = cta; ok && ti < n_items; ti += ncta) {
        const int vt = a.reverse ? cta + ncta * ((n_items - 1 - cta) / ncta) - (ti - cta) : ti;
        const int fr = vt / a.n_tiles, tile = vt - fr * a.n_tiles;
        const int tok0 = tile * a.tile_tokens;
        for (int kb = 0; kb < nkb; ++kb) {
          const long long w0 = tr ? clock64() : 0;
          ok = ptx::mbar_wait(&aempty[pa.stage], pa.phase ^ 1, a.dbg, kDbgProdEmpty | (unsigned)kb);
          if (!ok) break;
          if (tr) tw += clock64() - w0;
          const uint32_t sa = smem_base + Cfg::kAOff + pa.stage * 2 * kABytes;
          ptx::mbar_arrive_expect_tx(&afull[pa.stage], 2 * kABytes);
          const CUtensorMap *tm;
          int c0, row;
          if (kb < a.n_taps * a.kb_per_tap) {
            const int tap = kb / a.kb_per_tap;
            tm = &a.tm_ring;
            c0 = (kb - tap * a.kb_per_tap) * kBK;
            row = tcn_tap_row(a, fr, tap) + tok0;
          } else {
            tm = &a.tm_res;
            c0 = (kb - a.n_taps * a.kb_per_tap) * kBK;
            row = tcn_res_row(a, fr) + tok0;
          }
          // ring history and delayed residual are read once per step: stream them (evict-first) so the
          // frames written moments ago by the previous kernel stay in L2 until they are consumed
          ptx::tma_load_2d_hint(sa, tm, &afull[pa.stage], c0, row, ptx::kEvictFirst);
          ptx::tma_load_2d_hint(sa + kABytes, tm, &afull[pa.stage], c0, row + a.t_alloc, ptx::kEvictFirst);
          pa.advance<Cfg::kAStages>();
          ok = ptx::mbar_wait(&bempty[pb.stage], pb.phase ^ 1, a.dbg, kDbgProdEmpty | 0x800000u | (unsigned)kb);
          if (!ok) break;
          const uint32_t sb = smem_base + Cfg::kBOff + pb.stage * 2 * Cfg::kBBytes;
          ptx::mbar_arrive_expect_tx(&bfull[pb.stage], 2 * Cfg::kBBytes);
          ptx::tma_load_2d_hint(sb, &a.tm_w, &bfull[pb.stage], kb * kBK, 0, ptx::kEvictLast);
          ptx::tma_load_2d_hint(sb + Cfg::kBBytes, &a.tm_w, &bfull[pb.stage], kb * kBK, COUT, ptx::kEvictLast);
          pb.advance<Cfg::kBStages>();
        }
      }
      if (tr) {
        a.trace[24] = tw;
        a.trace[25] = clock64() - tstart;
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      PipeState pa, pb;
      bool ok = true;
      int it = 0;
      const bool tr = a.trace != nullptr && cta == 0;
      unsigned long long tw_ops = 0, tw_acc = 0;
      const long long tstart = tr ? clock64() : 0;
      for (int tile = cta; ok && tile < n_items; tile += ncta, ++it) {
        const int acc = it & 1;
        const long long w0 = tr ? clock64() : 0;
        ok = ptx::mbar_wait(&tempty[acc], ((it >> 1) & 1) ^ 1, a.dbg, kDbgMmaTmemEmpty | (unsigned)it);
        if (!ok) break;
        if (tr) tw_acc += clock64() - w0;
        ptx::tc_fence_after();
        const uint32_t d = tmem_base + acc * Cfg::kAccCols;
        for (int kb = 0; kb < nkb; ++kb) {
          const long long w1 = tr ? clock64() : 0;
          ok = ptx::mbar_wait(&afull[pa.stage], pa.phase, a.dbg, kDbgMmaFull | (unsigned)kb);
          if (!ok) break;
          ok = ptx::mbar_wait(&bfull[pb.stage], pb.phase, a.dbg, kDbgMmaFull | 0x800000u | (unsigned)kb);
          if (!ok) break;
          if (tr) tw_ops += clock64() - w1;
          ptx::tc_fence_after();
          const uint32_t sa = smem_base + Cfg::kAOff + pa.stage * 2 * kABytes;
          const uint32_t sb = smem_base + Cfg::kBOff + pb.stage * 2 * Cfg::kBBytes;
          if (Cfg::kStacked) issue_kblock_stacked<2 * COUT>(d, sa, sa + kABytes, sb, kb == 0);
          else issue_kblock<COUT>(d, sa, sa + kABytes, sb, sb + Cfg::kBBytes, kb == 0);
          ptx::umma_commit(&aempty[pa.stage]);
          ptx::umma_commit(&bempty[pb.stage]);
          pa.advance<Cfg::kAStages>();
          pb.advance<Cfg::kBStages>();
        }
        if (ok) ptx::umma_commit(&tfull[acc]);
      }
      if (tr) {
        a.trace[26] = tw_ops;
        a.trace[27] = tw_acc;
        a.trace[28] = clock64() - tstart;
      }
    }
  } else if (warp >= 4 && warp < 8) {
    const int q = warp & 3;
    bool ok = true;
    int it = 0;
    for (int ti = cta; ok && ti < n_items; ti += ncta, ++it) {
      const int vt = a.reverse ? cta + ncta * ((n_items - 1 - cta) / ncta) - (ti - cta) : ti;
      const int fr = vt / a.n_tiles, tile = vt - fr * a.n_tiles;
      const int acc = it & 1;
      ok = ptx::mbar_wait(&tfull[acc], (it >> 1) & 1, a.dbg, kDbgEpiTmemFull | (unsigned)it);
      if (!ok) break;
      ptx::tc_fence_after();
      const int row = q * 32 + lane;
      const long long tok = (long long)tile * a.tile_tokens + row;
      const bool valid = row < a.tile_tokens && tok < a.n_tokens;
      const EpiArgs epi = tcn_epi(a, fr);
      epilogue_rows<COUT, Cfg::kStacked>(tmem_base + ((uint32_t)(q * 32) << 16) + acc * Cfg::kAccCols, bias_s, epi, tok, valid);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tempty[acc]);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

template <int COUT>
__global__ void __launch_bounds__(256, 1) k_tc_tcn(const __grid_constant__ TcTcnArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  tcn_body<COUT>(a, smem_raw, (int)blockIdx.x, (int)gridDim.x);
}

// =============================================================================================
// temporal conv on CTA pairs (cta_group::2): the two CTAs of a cluster take two adjacent token
// tiles (UMMA M = 256) and each loads only half of every weight K-block (N/2 rows), which halves the
// weight bytes entering each SM and the weight shared-memory footprint -> deeper pipeline at COUT = 256.
// Protocol: "full" barriers live in the leader CTA and count the TMA bytes of BOTH CTAs; "empty" and
// "accumulator full" barriers exist in both CTAs and are signalled by multicast tcgen05.commit;
// "accumulator empty" lives in the leader and collects the epilogue warps of both CTAs.
// =============================================================================================
template <int COUT>
struct TcTcn2Cfg {
  static constexpr int kBHalfBytes = (COUT / 2) * kBK * 2;  // one plane, this CTA's half of the weight rows
  static constexpr int kAStages = 4;
  static constexpr int kBStages = COUT == 256 ? 3 : 4;
  static constexpr int kAOff = 0;
  static constexpr int kBOff = kAStages * 2 * kABytes;
  static constexpr int kBarOff = kBOff + kBStages * 2 * kBHalfBytes;
  static constexpr int kBiasOff = kBarOff + 256;
  static constexpr int kSmemBytes = kBiasOff + COUT * 4 + 1024;
  // stacked-B (see issue_kblock_stacked): CTA 0 of the pair holds the whole B_hi plane, CTA 1 the whole B_lo plane,
  // i.e. the two halves of the N' = 2*COUT operand rows that cta_group::2 splits across the pair
  static constexpr bool kStacked = COUT <= 128;
  static constexpr int kAccCols = kStacked ? 2 * COUT : COUT;
  static constexpr int kTmemCols = 2 * kAccCols;
  static_assert(kSmemBytes <= kSmemLimit, "shared memory budget");
};

template <int N2>
__device__ __forceinline__ void issue_kblock_pair_stacked(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_stack, bool first) {
  constexpr uint32_t idesc = ptx::umma_idesc_bf16(2 * kTileRows, N2);
  const uint32_t ah = ptx::umma_desc_lo(a_hi), al = ptx::umma_desc_lo(a_lo), bs = ptx::umma_desc_lo(b_stack);
#pragma unroll
  for (int k = 0; k < kBK / 16; ++k) {
    ptx::umma_bf16_pair_lo(tmem_d, ah + 2 * k, bs + 2 * k, idesc, (first && k == 0) ? 0u : 1u);
    ptx::umma_bf16_pair_lo(tmem_d, al + 2 * k, bs + 2 * k, idesc, 1u);
  }
}

template <int COUT>
__device__ __forceinline__ void issue_kblock_pair(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                                  bool first) {
  constexpr uint32_t idesc = ptx::umma_idesc_bf16(2 * kTileRows, COUT);
  const uint32_t ah = ptx::umma_desc_lo(a_hi), al = ptx::umma_desc_lo(a_lo), bh = ptx::umma_desc_lo(b_hi), bl = ptx::umma_desc_lo(b_lo);
#pragma unroll
  for (int k = 0; k < kBK / 16; ++k) {
    ptx::umma_bf16_pair_lo(tmem_d, ah + 2 * k, bh + 2 * k, idesc, (first && k == 0) ? 0u : 1u);
    ptx::umma_bf16_pair_lo(tmem_d, al + 2 * k, bh + 2 * k, idesc, 1u);
    ptx::umma_bf16_pair_lo(tmem_d, ah + 2 * k, bl + 2 * k, idesc, 1u);
  }
}

template <int COUT>
__device__ __forceinline__ void tcn2_body(const TcTcnArgs &a, uint8_t *smem_raw, const int cluster_id, const int n_clusters) {
  using Cfg = TcTcn2Cfg<COUT>;
  uint8_t *smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *afull = reinterpret_cast<uint64_t *>(smem + Cfg::kBarOff);
  uint64_t *aempty = afull + Cfg::kAStages;
  uint64_t *bfull = aempty + Cfg::kAStages;
  uint64_t *bempty = bfull + Cfg::kBStages;
  uint64_t *tfull = bempty + Cfg::kBStages;
  uint64_t *tempty = tfull + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + 2);
  float *bias_s = reinterpret_cast<float *>(smem + Cfg::kBiasOff);
  const uint32_t smem_base = ptx::smem_u32(smem);
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kAStages; ++s) {
      ptx::mbar_init(&afull[s], 1);
      ptx::mbar_init(&aempty[s], 1);
    }
    for (int s = 0; s < Cfg::kBStages; ++s) {
      ptx::mbar_init(&bfull[s], 1);
      ptx::mbar_init(&bempty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], 8);  // 4 epilogue warps of each CTA
    }
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&a.tm_ring);
    ptx::prefetch_tmap(&a.tm_w);
    if (a.kb_res) ptx::prefetch_tmap(&a.tm_res);
  }
  if (warp == 1) {
    ptx::tmem_alloc_pair(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish_pair();
  }
  for (int i = threadIdx.x; i < COUT; i += blockDim.x) bias_s[i] = a.epi.bias[i];
  ptx::tc_fence_before();
  ptx::cluster_sync_all();  // both CTAs' barriers are initialised before anything signals across the pair
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  const int nkb = a.n_taps * a.kb_per_tap + a.kb_res;
  const int pairs_per_frame = (a.n_tiles + 1) / 2;      // tile pairs never straddle two frames of a time-batched launch
  const int n_pairs = pairs_per_frame * a.n_frames;

  if (warp == 0) {
    if (lane == 0) {
      PipeState pa, pb;
      bool ok = true;
      for (int pi = cluster_id; ok && pi < n_pairs; pi += n_clusters) {
        const int vp = a.reverse ? cluster_id + n_clusters * ((n_pairs - 1 - cluster_id) / n_clusters) - (pi - cluster_id) : pi;
        const int fr = vp / pairs_per_frame, pr = vp - fr * pairs_per_frame;
        const int tok0 = (2 * pr + (int)rank) * a.tile_tokens;
        for (int kb = 0; kb < nkb; ++kb) {
          ok = ptx::mbar_wait(&aempty[pa.stage], pa.phase ^ 1, a.dbg, kDbgProdEmpty | (unsigned)kb);
          if (!ok) break;
          const uint32_t sa = smem_base + Cfg::kAOff + pa.stage * 2 * kABytes;
          if (leader) ptx::mbar_arrive_expect_tx(&afull[pa.stage], 2 * 2 * kABytes);  // bytes of both CTAs
          const uint32_t fa = ptx::mapa_u32(ptx::smem_u32(&afull[pa.stage]), 0);
          const CUtensorMap *tm;
          int c0, row;
          if (kb < a.n_taps * a.kb_per_tap) {
            const int tap = kb / a.kb_per_tap;
            tm = &a.tm_ring;
            c0 = (kb - tap * a.kb_per_tap) * kBK;
            row = tcn_tap_row(a, fr, tap) + tok0;
          } else {
            tm = &a.tm_res;
            c0 = (kb - a.n_taps * a.kb_per_tap) * kBK;
            row = tcn_res_row(a, fr) + tok0;
          }
          ptx::tma_load_2d_pair_hint(sa, tm, fa, c0, row, ptx::kEvictFirst);
          ptx::tma_load_2d_pair_hint(sa + kABytes, tm, fa, c0, row + a.t_alloc, ptx::kEvictFirst);
          pa.advance<Cfg::kAStages>();
          ok = ptx::mbar_wait(&bempty[pb.stage], pb.phase ^ 1, a.dbg, kDbgProdEmpty | 0x800000u | (unsigned)kb);
          if (!ok) break;
          const uint32_t sb = smem_base + Cfg::kBOff + pb.stage * 2 * Cfg::kBHalfBytes;
          if (leader) ptx::mbar_arrive_expect_tx(&bfull[pb.stage], 2 * 2 * Cfg::kBHalfBytes);
          const uint32_t fb = ptx::mapa_u32(ptx::smem_u32(&bfull[pb.stage]), 0);
          if (Cfg::kStacked) {
            // one box of COUT rows: the hi plane for CTA 0, the lo plane for CTA 1 (tm_w then has a COUT-row box)
            ptx::tma_load_2d_pair_hint(sb, &a.tm_w, fb, kb * kBK, (int)rank * COUT, ptx::kEvictLast);
          } else {
            ptx::tma_load_2d_pair_hint(sb, &a.tm_w, fb, kb * kBK, (int)rank * (COUT / 2), ptx::kEvictLast);
            ptx::tma_load_2d_pair_hint(sb + Cfg::kBHalfBytes, &a.tm_w, fb, kb * kBK, COUT + (int)rank * (COUT / 2), ptx::kEvictLast);
          }
          pb.advance<Cfg::kBStages>();
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {
      PipeState pa, pb;
      bool ok = true;
      int it = 0;
      for (int pr = cluster_id; ok && pr < n_pairs; pr += n_clusters, ++it) {
        const int acc = it & 1;
        ok = ptx::mbar_wait(&tempty[acc], ((it >> 1) & 1) ^ 1, a.dbg, kDbgMmaTmemEmpty | (unsigned)it);
        if (!ok) break;
        ptx::tc_fence_after();
        const uint32_t d = tmem_base + acc * Cfg::kAccCols;
        for (int kb = 0; kb < nkb; ++kb) {
          ok = ptx::mbar_wait(&afull[pa.stage], pa.phase, a.dbg, kDbgMmaFull | (unsigned)kb);
          if (!ok) break;
          ok = ptx::mbar_wait(&bfull[pb.stage], pb.phase, a.dbg, kDbgMmaFull | 0x800000u | (unsigned)kb);
          if (!ok) break;
          ptx::tc_fence_after();
          const uint32_t sa = smem_base + Cfg::kAOff + pa.stage * 2 * kABytes;
          const uint32_t sb = smem_base + Cfg::kBOff + pb.stage * 2 * Cfg::kBHalfBytes;
          if (Cfg::kStacked) issue_kblock_pair_stacked<2 * COUT>(d, sa, sa + kABytes, sb, kb == 0);
          else issue_kblock_pair<COUT>(d, sa, sa + kABytes, sb, sb + Cfg::kBHalfBytes, kb == 0);
          ptx::umma_commit_pair(&aempty[pa.stage], 3);
          ptx::umma_commit_pair(&bempty[pb.stage], 3);
          pa.advance<Cfg::kAStages>();
          pb.advance<Cfg::kBStages>();
        }
        if (ok) ptx::umma_commit_pair(&tfull[acc], 3);
      }
    }
  } else if (warp >= 4 && warp < 8) {
    const int q = warp & 3;
    bool ok = true;
    int it = 0;
    for (int pi = cluster_id; ok && pi < n_pairs; pi += n_clusters, ++it) {
      const int vp = a.reverse ? cluster_id + n_clusters * ((n_pairs - 1 - cluster_id) / n_clusters) - (pi - cluster_id) : pi;
      const int fr = vp / pairs_per_frame, pr = vp - fr * pairs_per_frame;
      const int acc = it & 1;
      ok = ptx::mbar_wait(&tfull[acc], (it >> 1) & 1, a.dbg, kDbgEpiTmemFull | (unsigned)it);
      if (!ok) break;
      ptx::tc_fence_after();
      const int tile = 2 * pr + (int)rank;
      const int row = q * 32 + lane;
      const long long tok = (long long)tile * a.tile_tokens + row;
      const bool valid = tile < a.n_tiles && row < a.tile_tokens && tok < a.n_tokens;
      const EpiArgs epi = tcn_epi(a, fr);
      epilogue_rows<COUT, Cfg::kStacked>(tmem_base + ((uint32_t)(q * 32) << 16) + acc * Cfg::kAccCols, bias_s, epi, tok, valid);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa_u32(ptx::smem_u32(&tempty[acc]), 0));
    }
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();  // nobody leaves (or frees TMEM) while the peer may still signal or read
  if (warp == 1) ptx::tmem_dealloc_pair(tmem_base, Cfg::kTmemCols);
}

template <int COUT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(256, 1) k_tc_tcn2(const __grid_constant__ TcTcnArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  tcn2_body<COUT>(a, smem_raw, (int)blockIdx.x / 2, (int)gridDim.x / 2);
}

// =============================================================================================
// graph conv: GEMM first, adjacency mix in the epilogue
//
//   z[w] = sum_i sum_v A_i[v,w] * (W_i x[v])  + gcn_residual(x)[w]      (models/base.py:262-269, by linearity)
//
// Per (tile, pass) work item the mainloop is a pure TMA -> tcgen05 pipeline computing
// Y = X [128 x cin] * [W_0 | W_1 | W_2 (| W_r)]^T for 64 output channels (N = P*64 accumulator columns;
// P = 4 when gcn_residual is a folded 1x1 conv, P = 3 when it is the identity).  The epilogue is split
// over two warp roles that hand 16-channel chunks over through shared memory with mbarriers:
//   drain warps (4, thread = token row): tcgen05.ld the chunk of every part, fold the own-row terms
//       T = a0[w]*Y0 (+ Y3) + bias, and write the planes T, Y1, Y2 (swizzled 64-byte rows);
//   mix warps (8, lane = channel, 2 token rows per instruction): z[w] = T[w] + sum over the CSR sources
//       of partitions 1 and 2 (+ identity residual row from global), ReLU, split, store.
// The transposed mix phase reads whole 64-byte row segments, so gathering arbitrary source rows is free
// of bank conflicts and of divergence, and the stores are sector-sized and contiguous.
// =============================================================================================

constexpr int kMixSlots = 6;    // non-zeros of partitions 1 and 2 together per output vertex
constexpr int kGcnChunk = 16;   // channels handed over per exchange buffer

struct TcGcnArgs {
  CUtensorMap tm_x;  // block input ring [kOutSlots*2*t_alloc rows][cin], box {64, 128}
  CUtensorMap tm_w;  // [2*P*cout rows][cin], box {64, P*64}; row = pass*(P*64) + part*64 + c; hi rows, then lo rows
  int x_row;         // first row of the hi plane of the input slot
  int t_alloc;
  int cin, cout;     // multiples of 64
  int V;
  int n_tiles, tile_tokens;
  long long n_tokens;
  const int *mix_ptr;  // CSR over (partition * V + output vertex); partition 0 must be diagonal (self links)
  const int *mix_src;
  const float *mix_val;
  unsigned long long *trace;  // optional phase timers written by CTA 0 (COSK_TRACE=1), else nullptr
  EpiArgs epi;                // r_hi/r_lo = input rows when cin == cout (identity gcn_residual, P = 3), else nullptr
  unsigned int *dbg;
  // adaptive graph conv (k_tc_agcn): per-token dense mixing rows written by the attention kernel,
  // dense[token*dense_ld + partition*dense_vp + source vertex]
  const float *dense;
  int dense_ld, dense_vp;
  // time-batched launch (n_frames > 1, plain graph conv only): frame f reads slot in_walk.slot(f) of the input ring and writes
  // slot out_walk.slot(f) of the temporal ring; epi.y_* / epi.r_* then point at slot 0 of their rings
  int n_frames = 1;
  int slot_rows = 0;
  RingWalk in_walk, out_walk;
  long long in_slot_elems = 0, out_slot_elems = 0;
};

__device__ __forceinline__ int gcn_x_row(const TcGcnArgs &a, int f) { return a.n_frames == 1 ? a.x_row : a.in_walk.slot(f) * a.slot_rows; }
__device__ __forceinline__ EpiArgs gcn_epi(const TcGcnArgs &a, int f) {
  EpiArgs e = a.epi;
  if (a.n_frames > 1) {
    const long long o = (long long)a.out_walk.slot(f) * a.out_slot_elems;
    e.y_hi += o;
    e.y_lo += o;
    if (e.r_hi != nullptr) {
      const long long r = (long long)a.in_walk.slot(f) * a.in_slot_elems;
      e.r_hi += r;
      e.r_lo += r;
    }
  }
  return e;
}

template <int P, int STAGES>
struct TcGcnCfg {
  // STAGES = 2: operand ring two K-blocks deep (cin >= 128: several K-blocks per work item).
  // STAGES = 1: a single operand stage -- enough when a work item is one K-block (cin = 64), because the
  //             next item's load + MMA fit inside the current item's epilogue -- and the shared memory
  //             saved buys four exchange buffers, so drain and mix warps run fully decoupled.
  static constexpr int kN = P * 64;
  static constexpr int kBBytes = kN * kBK * 2;
  static constexpr int kStageBytes = 2 * kABytes + 2 * kBBytes;
  static constexpr int kStages = STAGES;
  static constexpr int kPlaneBytes = kTileRows * kGcnChunk * 4;  // 8 KB: 128 rows x 16 floats
  static constexpr int kExchBytes = 3 * kPlaneBytes;             // planes T, Y1, Y2
  static constexpr int kExchBufs = STAGES == 1 ? 4 : (P == 3 ? 2 : 1);
  static constexpr int kExchOff = kStages * kStageBytes;
  static constexpr int kCsrOff = kExchOff + kExchBufs * kExchBytes;  // per row: n, coef[slots], src[slots], row order
  static constexpr int kCsrBytes = kTileRows * (4 + 4 * kMixSlots) + kTileRows * 8;
  static constexpr int kBarOff = kCsrOff + kCsrBytes;
  static constexpr int kBiasOff = kBarOff + 256;
  static constexpr int kSmemBytes = kBiasOff + 256 * 4 + 1024;
  static constexpr int kAccStride = 256;
  static constexpr int kTmemCols = 512;
  static_assert(kSmemBytes <= kSmemLimit, "shared memory budget");
  static_assert(kExchBufs <= 4, "exchange barriers");
};

// byte offset of element (row, col) in an exchange plane: 64-byte rows, 16-byte chunks XOR-swizzled with
// (row >> 1) so that 8 consecutive rows writing the same chunk, and any two rows of different parity
// reading whole rows, never meet in a bank
__device__ __forceinline__ uint32_t exch_off(int row, int chunk) { return row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4); }

// Mix-phase gather of one 16-channel chunk for the two row groups of a lane, with the slot count N known
// at compile time: all shared-memory loads are issued before the first FMA (no branch per slot), unused
// slots of a row carry a zero coefficient and offset 0.
template <int N>
__device__ __forceinline__ void mix_gather(const uint8_t *buf, const uint32_t (&off_t)[2], const uint32_t (&off_s)[2][kMixSlots / 2],
                                           const float (&cf)[2][kMixSlots], float4 (&z)[2]) {
  float4 y[2][N > 0 ? N : 1];
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    z[g] = *reinterpret_cast<const float4 *>(buf + off_t[g]);
#pragma unroll
    for (int e = 0; e < N; ++e) {
      const uint32_t off = (e & 1) ? (off_s[g][e >> 1] >> 16) : (off_s[g][e >> 1] & 0xffffu);
      y[g][e] = *reinterpret_cast<const float4 *>(buf + off);
    }
  }
#pragma unroll
  for (int e = 0; e < N; ++e) {
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      z[g].x = fmaf(cf[g][e], y[g][e].x, z[g].x);
      z[g].y = fmaf(cf[g][e], y[g][e].y, z[g].y);
      z[g].z = fmaf(cf[g][e], y[g][e].z, z[g].z);
      z[g].w = fmaf(cf[g][e], y[g][e].w, z[g].w);
    }
  }
}

// TMA producer of the graph-conv kernels (one elected thread): per (tile, pass, K-block) the input tile rows
// (hi, lo) and the [P*64 x 64] weight slab (hi, lo) of that pass.
template <class Cfg, int P>
__device__ __forceinline__ void gcn_producer(const TcGcnArgs &a, uint64_t *full, uint64_t *empty, const uint32_t smem_base,
                                             const int cta, const int ncta) {
  const int n_pass = a.cout / 64;
  const int nkb = a.cin / kBK;
  PipeState ps;
  bool ok = true;
  for (int vt = cta; ok && vt < a.n_tiles * a.n_frames; vt += ncta) {
    const int fr = vt / a.n_tiles, tile = vt - fr * a.n_tiles;
    const int row = gcn_x_row(a, fr) + tile * a.tile_tokens;
    for (int pass = 0; ok && pass < n_pass; ++pass) {
      for (int kc = 0; kc < nkb; ++kc) {
        ok = ptx::mbar_wait(&empty[ps.stage], ps.phase ^ 1, a.dbg, kDbgProdEmpty | (unsigned)(pass * 16 + kc));
        if (!ok) break;
        const uint32_t st = smem_base + ps.stage * Cfg::kStageBytes;
        ptx::mbar_arrive_expect_tx(&full[ps.stage], Cfg::kStageBytes);
        // the input tile is re-read once per pass (L2 hits): keep it until the last pass, then let it go
        const uint64_t xpol = pass + 1 < n_pass ? ptx::kEvictNormal : ptx::kEvictFirst;
        ptx::tma_load_2d_hint(st, &a.tm_x, &full[ps.stage], kc * kBK, row, xpol);
        ptx::tma_load_2d_hint(st + kABytes, &a.tm_x, &full[ps.stage], kc * kBK, row + a.t_alloc, xpol);
        ptx::tma_load_2d_hint(st + 2 * kABytes, &a.tm_w, &full[ps.stage], kc * kBK, pass * Cfg::kN, ptx::kEvictLast);
        ptx::tma_load_2d_hint(st + 2 * kABytes + Cfg::kBBytes, &a.tm_w, &full[ps.stage], kc * kBK, P * a.cout + pass * Cfg::kN,
                              ptx::kEvictLast);
        ps.advance<Cfg::kStages>();
      }
    }
  }
}

// MMA issuer of the graph-conv kernels (one elected thread): one accumulator of Cfg::kN columns per
// (tile, pass), double buffered in TMEM.
template <class Cfg, bool TRACE>
__device__ __forceinline__ void gcn_mma_issuer(const TcGcnArgs &a, uint64_t *full, uint64_t *empty, uint64_t *tfull, uint64_t *tempty,
                                               const uint32_t smem_base, const uint32_t tmem_base, const int cta, const int ncta) {
  const int n_pass = a.cout / 64;
  const int nkb = a.cin / kBK;
  PipeState ps;
  bool ok = true;
  int it = 0;
  const bool mtr = TRACE && a.trace != nullptr && cta == 0;
  unsigned long long mt[2] = {0, 0};
  const long long mstart = mtr ? clock64() : 0;
  for (int tile = cta; ok && tile < a.n_tiles * a.n_frames; tile += ncta) {
    for (int pass = 0; ok && pass < n_pass; ++pass, ++it) {
      const int acc = it & 1;
      const long long m0 = mtr ? clock64() : 0;
      ok = ptx::mbar_wait(&tempty[acc], ((it >> 1) & 1) ^ 1, a.dbg, kDbgMmaTmemEmpty | (unsigned)it);
      if (!ok) break;
      if (mtr) mt[0] += clock64() - m0;
      ptx::tc_fence_after();
      const uint32_t d = tmem_base + acc * Cfg::kAccStride;
      for (int kc = 0; kc < nkb; ++kc) {
        const long long m1 = mtr ? clock64() : 0;
        ok = ptx::mbar_wait(&full[ps.stage], ps.phase, a.dbg, kDbgMmaFull | (unsigned)(pass * 16 + kc));
        if (!ok) break;
        if (mtr) mt[1] += clock64() - m1;
        ptx::tc_fence_after();
        const uint32_t st = smem_base + ps.stage * Cfg::kStageBytes;
        issue_kblock<Cfg::kN>(d, st, st + kABytes, st + 2 * kABytes, st + 2 * kABytes + Cfg::kBBytes, kc == 0);
        ptx::umma_commit(&empty[ps.stage]);
        ps.advance<Cfg::kStages>();
      }
      if (ok) ptx::umma_commit(&tfull[acc]);
    }
  }
  if (mtr) {
    a.trace[16] = mt[0];
    a.trace[17] = mt[1];
    a.trace[18] = clock64() - mstart;
  }
}

template <int P, int STAGES, bool TRACE>
__device__ __forceinline__ void gcn_body(const TcGcnArgs &a, uint8_t *smem_raw, const int cta, const int ncta) {
  using Cfg = TcGcnCfg<P, STAGES>;
  uint8_t *smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *full = reinterpret_cast<uint64_t *>(smem + Cfg::kBarOff);
  uint64_t *empty = full + Cfg::kStages;
  uint64_t *tfull = empty + Cfg::kStages;
  uint64_t *tempty = tfull + 2;
  uint64_t *xfull = tempty + 2;
  uint64_t *xempty = xfull + 4;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(xempty + 4);
  float *bias_s = reinterpret_cast<float *>(smem + Cfg::kBiasOff);
  // CSR of partitions 1 and 2 per tile row, shared by the mix warps
  int *csr_n = reinterpret_cast<int *>(smem + Cfg::kCsrOff);                 // [128]
  float *csr_coef = reinterpret_cast<float *>(csr_n + kTileRows);             // [8][128]
  uint8_t *csr_src = reinterpret_cast<uint8_t *>(csr_coef + kMixSlots * kTileRows);  // [slots][128]: plane (bit 7) | source row
  uint8_t *csr_perm = csr_src + kMixSlots * kTileRows;                               // [128] mix-phase row order
  const uint32_t smem_base = ptx::smem_u32(smem);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], 4);  // the four drain warps
    }
    for (int s = 0; s < Cfg::kExchBufs; ++s) {
      ptx::mbar_init(&xfull[s], 4);   // the four drain warps
      ptx::mbar_init(&xempty[s], 8);  // the eight mix warps
    }
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&a.tm_x);
    ptx::prefetch_tmap(&a.tm_w);
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish();
  }
  for (int i = threadIdx.x; i < a.cout; i += blockDim.x) bias_s[i] = a.epi.bias[i];
  if (threadIdx.x < kTileRows) {
    const int row = threadIdx.x;
    const int wv = row % a.V, sk0 = row - wv;
    int n = 0;
    for (int e = 0; e < kMixSlots; ++e) {
      csr_coef[e * kTileRows + row] = 0.f;
      csr_src[e * kTileRows + row] = 0;
    }
    if (row < a.tile_tokens) {
      for (int p = 1; p < 3; ++p)
        for (int e = a.mix_ptr[p * a.V + wv]; e < a.mix_ptr[p * a.V + wv + 1] && n < kMixSlots; ++e) {
          csr_coef[n * kTileRows + row] = a.mix_val[e];
          csr_src[n * kTileRows + row] = (uint8_t)(((p - 1) << 7) | (sk0 + a.mix_src[e]));
          ++n;
        }
    }
    csr_n[row] = n;
  }
  __syncthreads();
  if (threadIdx.x < kTileRows) {
    // rank of this row when rows are ordered by descending source count (ties by row index): the mix
    // warps walk rows in that order, so the 8 rows sharing an instruction need about the same slots
    const int row = threadIdx.x, n = csr_n[row];
    int rank = 0;
    for (int r = 0; r < kTileRows; ++r) {
      const int nr = csr_n[r];
      rank += (nr > n || (nr == n && r < row)) ? 1 : 0;
    }
    csr_perm[rank] = (uint8_t)row;
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();  // prologue above touched only static data; activations of the previous kernel from here on
  const int n_pass = a.cout / 64;
  constexpr int kChunks = 64 / kGcnChunk;

  if (warp == 0) {
    if (lane == 0) gcn_producer<Cfg, P>(a, full, empty, smem_base, cta, ncta);
  } else if (warp == 1) {
    if (lane == 0) gcn_mma_issuer<Cfg, TRACE>(a, full, empty, tfull, tempty, smem_base, tmem_base, cta, ncta);
  } else if (warp >= 4 && warp < 8) {
    // ---- drain: TMEM -> own-row terms folded -> exchange planes --------------------------------
    const int q = warp & 3;
    const int row = q * 32 + lane;
    float d0 = 0.f;  // coefficient of the self link (partition 0 is diagonal)
    if (row < a.tile_tokens) {
      const int wv = row % a.V;
      const int e0 = a.mix_ptr[wv];
      if (a.mix_ptr[wv + 1] > e0) d0 = a.mix_val[e0];
    }
    const bool tr = TRACE && a.trace != nullptr && cta == 0 && q == 0 && lane == 0;
    unsigned long long tr_t[4] = {0, 0, 0, 0};
    long long tr_c = 0;
    const long long tr_start = tr ? clock64() : 0;
    bool ok = true;
    int it = 0;
    uint32_t xc = 0;  // exchange chunks handed over so far
    const int n_items = a.n_tiles * a.n_frames;  // (frame, tile) work items of a time-batched launch
    for (int tile = cta; ok && tile < n_items; tile += ncta) {
      for (int pass = 0; ok && pass < n_pass; ++pass, ++it) {
        const int acc = it & 1;
        if (tr) tr_c = clock64();
        ok = ptx::mbar_wait(&tfull[acc], (it >> 1) & 1, a.dbg, kDbgEpiTmemFull | (unsigned)it);
        if (!ok) break;
        if (tr) { const long long n_ = clock64(); tr_t[0] += n_ - tr_c; tr_c = n_; }
        ptx::tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * Cfg::kAccStride;
#pragma unroll 1
        for (int c = 0; c < kChunks; ++c, ++xc) {
          const int c0 = pass * 64 + c * kGcnChunk;
          float t[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) t[j] = bias_s[c0 + j];
          uint32_t y0[16], y1[16], y2[16];
          ptx::tmem_ld_32x16(taddr + 0 * 64 + c * kGcnChunk, y0);
          ptx::tmem_ld_32x16(taddr + 1 * 64 + c * kGcnChunk, y1);
          ptx::tmem_ld_32x16(taddr + 2 * 64 + c * kGcnChunk, y2);
          if (P == 4) {
            uint32_t y3[16];
            ptx::tmem_ld_32x16(taddr + 3 * 64 + c * kGcnChunk, y3);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) t[j] += __uint_as_float(y3[j]);
          } else {
            ptx::tmem_ld_wait();
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) t[j] = fmaf(d0, __uint_as_float(y0[j]), t[j]);
          if (tr) { const long long n_ = clock64(); tr_t[1] += n_ - tr_c; tr_c = n_; }
          const uint32_t b = xc % Cfg::kExchBufs;
          const uint32_t use = xc / Cfg::kExchBufs;
          ok = ptx::mbar_wait(&xempty[b], (use & 1) ^ 1, a.dbg, kDbgEpiExchEmpty | (xc & 0xffff));
          if (!ok) break;
          if (tr) { const long long n_ = clock64(); tr_t[2] += n_ - tr_c; tr_c = n_; }
          uint8_t *buf = smem + Cfg::kExchOff + b * Cfg::kExchBytes;
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) {
            const uint32_t off = exch_off(row, ch);
            *reinterpret_cast<float4 *>(buf + off) = make_float4(t[4 * ch], t[4 * ch + 1], t[4 * ch + 2], t[4 * ch + 3]);
            *reinterpret_cast<uint4 *>(buf + Cfg::kPlaneBytes + off) = make_uint4(y1[4 * ch], y1[4 * ch + 1], y1[4 * ch + 2], y1[4 * ch + 3]);
            *reinterpret_cast<uint4 *>(buf + 2 * Cfg::kPlaneBytes + off) = make_uint4(y2[4 * ch], y2[4 * ch + 1], y2[4 * ch + 2], y2[4 * ch + 3]);
          }
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&xfull[b]);
          if (tr) { const long long n_ = clock64(); tr_t[3] += n_ - tr_c; tr_c = n_; }
        }
        if (!ok) break;
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&tempty[acc]);  // accumulator fully read: the MMA may overwrite it
      }
    }
    if (tr) {
      for (int i = 0; i < 4; ++i) a.trace[i] = tr_t[i];
      a.trace[5] = clock64() - tr_start;
      a.trace[6] = (unsigned long long)it;
    }
  } else if (warp >= 8) {
    // ---- mix: one instruction covers 8 token rows x 16 channels (lane = row, 4-channel quad) -----------
    // A lane always serves the same 2 tile rows (tiles are skeleton aligned), so the byte offsets of its
    // CSR sources inside an exchange buffer are computed once and live in registers; rows are walked in
    // the count-sorted order, and (row group, slot) pairs empty for all 8 rows are skipped warp-uniformly.
    const int m = warp - 8;
    const int rr = lane >> 2, cq = lane & 3;
    int rows[2];
    uint32_t off_t[2], off_s[2][kMixSlots / 2];
    float cf[2][kMixSlots];
    int nmax = 0;  // most slots any of this warp's 16 rows needs (warp-uniform; rows are count-sorted, so mostly 1-2)
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      const int row = csr_perm[m * 16 + g * 8 + rr];
      rows[g] = row;
      off_t[g] = exch_off(row, cq);
      const int n = csr_n[row];
      nmax = max(nmax, n);
#pragma unroll
      for (int e = 0; e < kMixSlots; ++e) {
        const bool on = e < n;
        const uint32_t sp = on ? csr_src[e * kTileRows + row] : 0u;
        const uint32_t off = on ? (1 + (sp >> 7)) * Cfg::kPlaneBytes + exch_off((int)(sp & 0x7f), cq) : 0u;
        if (e & 1) off_s[g][e >> 1] |= off << 16;
        else off_s[g][e >> 1] = off;
        cf[g][e] = on ? csr_coef[e * kTileRows + row] : 0.f;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, o));
    const bool tr = TRACE && a.trace != nullptr && cta == 0 && m == 0 && lane == 0;
    unsigned long long tr_t[3] = {0, 0, 0};
    long long tr_c = 0;
    bool ok = true;
    uint32_t xc = 0;
    for (int vt = cta; ok && vt < a.n_tiles * a.n_frames; vt += ncta) {
      const int fr = vt / a.n_tiles, tile = vt - fr * a.n_tiles;
      const long long tok0 = (long long)tile * a.tile_tokens;
      const EpiArgs epi = gcn_epi(a, fr);
      for (int pass = 0; ok && pass < n_pass; ++pass) {
#pragma unroll 1
        for (int c = 0; c < kChunks; ++c, ++xc) {
          const int c0 = pass * 64 + c * kGcnChunk + 4 * cq;
          const uint32_t b = xc % Cfg::kExchBufs;
          const uint32_t use = xc / Cfg::kExchBufs;
          // identity gcn_residual added here (P == 3 and not folded into W_0): the two rows' 4 channels, issued before the wait
          uint2 rh[2] = {make_uint2(0, 0), make_uint2(0, 0)}, rl[2] = {make_uint2(0, 0), make_uint2(0, 0)};
          if (P == 3 && a.epi.r_hi != nullptr) {
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              const long long tok = tok0 + rows[g];
              if (rows[g] < a.tile_tokens && tok < a.n_tokens) {
                rh[g] = __ldg(reinterpret_cast<const uint2 *>(epi.r_hi + tok * epi.cs_r + c0));
                rl[g] = __ldg(reinterpret_cast<const uint2 *>(epi.r_lo + tok * epi.cs_r + c0));
              }
            }
          }
          if (tr) tr_c = clock64();
          ok = ptx::mbar_wait(&xfull[b], use & 1, a.dbg, kDbgEpiExchFull | (xc & 0xffff));
          if (!ok) break;
          if (tr) { const long long n_ = clock64(); tr_t[0] += n_ - tr_c; tr_c = n_; }
          const uint8_t *buf = smem + Cfg::kExchOff + b * Cfg::kExchBytes;
          float4 z[2];
          switch (nmax) {
            case 0: mix_gather<0>(buf, off_t, off_s, cf, z); break;
            case 1: mix_gather<1>(buf, off_t, off_s, cf, z); break;
            case 2: mix_gather<2>(buf, off_t, off_s, cf, z); break;
            case 3: mix_gather<3>(buf, off_t, off_s, cf, z); break;
            case 4: mix_gather<4>(buf, off_t, off_s, cf, z); break;
            case 5: mix_gather<5>(buf, off_t, off_s, cf, z); break;
            default: mix_gather<6>(buf, off_t, off_s, cf, z); break;
          }
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&xempty[b]);  // planes consumed: the drain warps may refill them
          if (P == 3 && a.epi.r_hi != nullptr) {
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              z[g].x += bf16_lo_as_float(rh[g].x) + bf16_lo_as_float(rl[g].x);
              z[g].y += bf16_hi_as_float(rh[g].x) + bf16_hi_as_float(rl[g].x);
              z[g].z += bf16_lo_as_float(rh[g].y) + bf16_lo_as_float(rl[g].y);
              z[g].w += bf16_hi_as_float(rh[g].y) + bf16_hi_as_float(rl[g].y);
            }
          }
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            const long long tok = tok0 + rows[g];
            if (rows[g] < a.tile_tokens && tok < a.n_tokens) {
              const float x0 = fmaxf(z[g].x, 0.f), x1 = fmaxf(z[g].y, 0.f), x2 = fmaxf(z[g].z, 0.f), x3 = fmaxf(z[g].w, 0.f);
              const uint32_t h0 = pack_bf16x2(x0, x1), h1 = pack_bf16x2(x2, x3);
              const uint32_t l0 = pack_bf16x2(x0 - bf16_lo_as_float(h0), x1 - bf16_hi_as_float(h0));
              const uint32_t l1 = pack_bf16x2(x2 - bf16_lo_as_float(h1), x3 - bf16_hi_as_float(h1));
              *reinterpret_cast<uint2 *>(epi.y_hi + tok * epi.cs_out + c0) = make_uint2(h0, h1);
              *reinterpret_cast<uint2 *>(epi.y_lo + tok * epi.cs_out + c0) = make_uint2(l0, l1);
            }
          }
          if (tr) { const long long n_ = clock64(); tr_t[1] += n_ - tr_c; tr_c = n_; }
        }
      }
    }
    if (tr) {
      a.trace[8] = tr_t[0];
      a.trace[9] = tr_t[1];
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

template <int P, int STAGES, bool TRACE>
__global__ void __launch_bounds__(512, 1) k_tc_gcn(const __grid_constant__ TcGcnArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  gcn_body<P, STAGES, TRACE>(a, smem_raw, (int)blockIdx.x, (int)gridDim.x);
}

// =============================================================================================
// Adaptive graph conv, GEMM + dense mix (AdaptiveGraphConvolution, models/a_gcn/a_gcn.py:52-69 with T = 1):
//
//   z[w] = sum_i sum_v M_i[v,w] * (W_i x[v]) + bias + gcn_residual(x)[w] ,   M_i = softmax_i + A_i + graph_attn_i
//
// Same TMA -> tcgen05 mainloop as k_tc_gcn (Y = X [W_0|W_1|W_2(|W_r)]^T, 64 output channels per pass), but the
// mixing matrix is dense and differs per skeleton, so the epilogue changes:
//   drain warps (4, thread = token row): copy 16-channel chunks of every part from TMEM to shared-memory planes
//       (80-byte rows: conflict-free 16-byte stores, and sources are immediate offsets from a lane's skeleton);
//   mix warps (8, lane = token row x 8-channel half): the 3*V coefficients of the lane's row sit in registers for
//       the whole tile (loaded from the scratch k_tc_attn / k_agcn_attn wrote), every source row is a broadcast
//       shared-memory read, 8 FMAs per 2 loads: the phase is bound by the FP32 pipe.
// P = 4: part 3 = folded gcn_residual conv (added from its plane); P = 3: identity residual added from the input rows.
// =============================================================================================
template <int P, int STAGES>
struct TcAgcnCfg {
  static constexpr int kN = P * 64;
  static constexpr int kBBytes = kN * kBK * 2;
  static constexpr int kStageBytes = 2 * kABytes + 2 * kBBytes;
  static constexpr int kStages = STAGES;
  static constexpr int kRowBytes = kGcnChunk * 4 + 16;           // 64-byte rows padded to 80
  static constexpr int kPlaneBytes = kTileRows * kRowBytes;      // 10 KB
  static constexpr int kExchBytes = P * kPlaneBytes;             // planes Y0, Y1, Y2 (, Y3)
  static constexpr int kExchBufs = 2;
  static constexpr int kExchOff = kStages * kStageBytes;
  static constexpr int kBarOff = kExchOff + kExchBufs * kExchBytes;
  static constexpr int kBiasOff = kBarOff + 256;
  static constexpr int kSmemBytes = kBiasOff + 256 * 4 + 1024;
  static constexpr int kAccStride = 256;
  static constexpr int kTmemCols = 512;
  static_assert(kSmemBytes <= kSmemLimit, "shared memory budget");
};

template <int P, int STAGES, int V>
__device__ __forceinline__ void agcn_body(const TcGcnArgs &a, uint8_t *smem_raw, const int cta, const int ncta) {
  using Cfg = TcAgcnCfg<P, STAGES>;
  constexpr int VP = (V + 3) / 4 * 4;  // == dense_vp
  uint8_t *smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *full = reinterpret_cast<uint64_t *>(smem + Cfg::kBarOff);
  uint64_t *empty = full + Cfg::kStages;
  uint64_t *tfull = empty + Cfg::kStages;
  uint64_t *tempty = tfull + 2;
  uint64_t *xfull = tempty + 2;
  uint64_t *xempty = xfull + Cfg::kExchBufs;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(xempty + Cfg::kExchBufs);
  float *bias_s = reinterpret_cast<float *>(smem + Cfg::kBiasOff);
  const uint32_t smem_base = ptx::smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], 4);
    }
    for (int s = 0; s < Cfg::kExchBufs; ++s) {
      ptx::mbar_init(&xfull[s], 4);
      ptx::mbar_init(&xempty[s], 8);
    }
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&a.tm_x);
    ptx::prefetch_tmap(&a.tm_w);
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish();
  }
  for (int i = threadIdx.x; i < a.cout; i += blockDim.x) bias_s[i] = a.epi.bias[i];
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  const int n_pass = a.cout / 64;
  constexpr int kChunks = 64 / kGcnChunk;

  if (warp == 0) {
    if (lane == 0) gcn_producer<Cfg, P>(a, full, empty, smem_base, cta, ncta);
  } else if (warp == 1) {
    if (lane == 0) gcn_mma_issuer<Cfg, false>(a, full, empty, tfull, tempty, smem_base, tmem_base, cta, ncta);
  } else if (warp >= 4 && warp < 8) {
    // ---- drain: TMEM -> exchange planes, no arithmetic -----------------------------------------
    const int q = warp & 3;
    const int row = q * 32 + lane;
    bool ok = true;
    int it = 0;
    uint32_t xc = 0;
    for (int tile = cta; ok && tile < a.n_tiles; tile += ncta) {
      for (int pass = 0; ok && pass < n_pass; ++pass, ++it) {
        const int acc = it & 1;
        ok = ptx::mbar_wait(&tfull[acc], (it >> 1) & 1, a.dbg, kDbgEpiTmemFull | (unsigned)it);
        if (!ok) break;
        ptx::tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * Cfg::kAccStride;
#pragma unroll 1
        for (int c = 0; c < kChunks; ++c, ++xc) {
          uint32_t y[P][16];
#pragma unroll
          for (int part = 0; part < P; ++part) ptx::tmem_ld_32x16(taddr + part * 64 + c * kGcnChunk, y[part]);
          ptx::tmem_ld_wait();
          const uint32_t b = xc % Cfg::kExchBufs;
          const uint32_t use = xc / Cfg::kExchBufs;
          ok = ptx::mbar_wait(&xempty[b], (use & 1) ^ 1, a.dbg, kDbgEpiExchEmpty | (xc & 0xffff));
          if (!ok) break;
          uint8_t *buf = smem + Cfg::kExchOff + b * Cfg::kExchBytes + row * Cfg::kRowBytes;
#pragma unroll
          for (int part = 0; part < P; ++part)
#pragma unroll
            for (int ch = 0; ch < 4; ++ch)
              *reinterpret_cast<uint4 *>(buf + part * Cfg::kPlaneBytes + ch * 16) =
                  make_uint4(y[part][4 * ch], y[part][4 * ch + 1], y[part][4 * ch + 2], y[part][4 * ch + 3]);
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&xfull[b]);
        }
        if (!ok) break;
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&tempty[acc]);
      }
    }
  } else if (warp >= 8) {
    // ---- dense mix ---------------------------------------------------------------------------------
    const int m = warp - 8;
    const int row = m * 16 + (lane >> 1), half = lane & 1;
    const bool row_ok = row < a.tile_tokens;
    const int sk0 = row_ok ? row - row % V : 0;  // first row of the lane's skeleton
    const uint32_t src_off = (uint32_t)(sk0 * Cfg::kRowBytes + half * 32);  // source vertex v adds v * kRowBytes
    const uint32_t own_off = (uint32_t)(row * Cfg::kRowBytes + half * 32);
    bool ok = true;
    uint32_t xc = 0;
    for (int tile = cta; ok && tile < a.n_tiles; tile += ncta) {
      const long long tok = (long long)tile * a.tile_tokens + row;
      const bool valid = row_ok && tok < a.n_tokens;
      // mixing row of this token: 3 partitions x V sources, in registers for the whole tile
      float4 cf[3][VP / 4];
#pragma unroll
      for (int part = 0; part < 3; ++part)
#pragma unroll
        for (int j = 0; j < VP / 4; ++j)
          cf[part][j] = valid ? *reinterpret_cast<const float4 *>(a.dense + tok * a.dense_ld + part * VP + 4 * j) : make_float4(0.f, 0.f, 0.f, 0.f);
      for (int pass = 0; ok && pass < n_pass; ++pass) {
#pragma unroll 1
        for (int c = 0; c < kChunks; ++c, ++xc) {
          const int c0 = pass * 64 + c * kGcnChunk + half * 8;
          float z[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) z[j] = bias_s[c0 + j];
          if (P == 3 && valid) {  // identity gcn_residual: the token's own input row (hi + lo)
            const uint4 h = ptx::ldg_v4(reinterpret_cast<const uint4 *>(a.epi.r_hi + tok * a.epi.cs_r + c0));
            const uint4 l = ptx::ldg_v4(reinterpret_cast<const uint4 *>(a.epi.r_lo + tok * a.epi.cs_r + c0));
            const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              z[2 * w] += bf16_lo_as_float(hw[w]) + bf16_lo_as_float(lw[w]);
              z[2 * w + 1] += bf16_hi_as_float(hw[w]) + bf16_hi_as_float(lw[w]);
            }
          }
          const uint32_t b = xc % Cfg::kExchBufs;
          const uint32_t use = xc / Cfg::kExchBufs;
          ok = ptx::mbar_wait(&xfull[b], use & 1, a.dbg, kDbgEpiExchFull | (xc & 0xffff));
          if (!ok) break;
          const uint8_t *buf = smem + Cfg::kExchOff + b * Cfg::kExchBytes;
          if (P == 4) {
            const float4 r0 = *reinterpret_cast<const float4 *>(buf + 3 * Cfg::kPlaneBytes + own_off);
            const float4 r1 = *reinterpret_cast<const float4 *>(buf + 3 * Cfg::kPlaneBytes + own_off + 16);
            z[0] += r0.x; z[1] += r0.y; z[2] += r0.z; z[3] += r0.w;
            z[4] += r1.x; z[5] += r1.y; z[6] += r1.z; z[7] += r1.w;
          }
#pragma unroll
          for (int part = 0; part < 3; ++part) {
            const uint8_t *pl = buf + part * Cfg::kPlaneBytes + src_off;
#pragma unroll
            for (int v = 0; v < V; ++v) {
              const float4 q4 = cf[part][v >> 2];
              const float coef = (v & 3) == 0 ? q4.x : (v & 3) == 1 ? q4.y : (v & 3) == 2 ? q4.z : q4.w;
              const float4 y0 = *reinterpret_cast<const float4 *>(pl + v * Cfg::kRowBytes);
              const float4 y1 = *reinterpret_cast<const float4 *>(pl + v * Cfg::kRowBytes + 16);
              z[0] = fmaf(coef, y0.x, z[0]); z[1] = fmaf(coef, y0.y, z[1]); z[2] = fmaf(coef, y0.z, z[2]); z[3] = fmaf(coef, y0.w, z[3]);
              z[4] = fmaf(coef, y1.x, z[4]); z[5] = fmaf(coef, y1.y, z[5]); z[6] = fmaf(coef, y1.z, z[6]); z[7] = fmaf(coef, y1.w, z[7]);
            }
          }
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&xempty[b]);
          if (valid) {
            uint32_t oh[4], ol[4];
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              const float x0 = fmaxf(z[2 * w], 0.f), x1 = fmaxf(z[2 * w + 1], 0.f);
              oh[w] = pack_bf16x2(x0, x1);
              ol[w] = pack_bf16x2(x0 - bf16_lo_as_float(oh[w]), x1 - bf16_hi_as_float(oh[w]));
            }
            *reinterpret_cast<uint4 *>(a.epi.y_hi + tok * a.epi.cs_out + c0) = make_uint4(oh[0], oh[1], oh[2], oh[3]);
            *reinterpret_cast<uint4 *>(a.epi.y_lo + tok * a.epi.cs_out + c0) = make_uint4(ol[0], ol[1], ol[2], ol[3]);
          }
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

template <int P, int STAGES, int V>
__global__ void __launch_bounds__(512, 1) k_tc_agcn(const __grid_constant__ TcGcnArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  agcn_body<P, STAGES, V>(a, smem_raw, (int)blockIdx.x, (int)gridDim.x);
}

// =============================================================================================
// Adaptive graph conv, attention half on tcgen05 (AdaptiveGraphConvolution.forward with T = 1,
// models/a_gcn/a_gcn.py:52-63).  Work item = (token tile, partition i):
//   mainloop   [theta_i | phi_i] = X [128 x cin] * [Wa_i | Wb_i]^T, 2*IC columns, stacked-B split products
//              (the hi and lo weight rows of a partition are adjacent in memory: one operand of 4*IC rows);
//   epilogue   (2 groups of 4 warps on alternate items, thread = token row) accumulator -> shared memory (theta in a skeleton-padded
//              layout so a lane reads its skeleton's V values with 16-byte broadcast loads), then per row w:
//              S[v] = <theta[v], phi[w]> / IC, softmax over v, + (A + graph_attn)_i[v][w], written as the
//              token's mixing row to the dense scratch k_tc_agcn reads.
// Group g owns TMEM accumulator g, so two items are in their epilogue while the MMAs of a third are issued.
// =============================================================================================
struct TcAttnArgs {
  CUtensorMap tm_x;  // block input ring, box {64, 128}
  CUtensorMap tm_w;  // [3 partitions][hi: theta, phi | lo: theta, phi][cin], box {64, 4*IC}
  int x_row, t_alloc, cin;
  int n_tiles, tile_tokens;
  long long n_tokens;
  const float *bias;  // [3][2*IC]
  const float *adj;   // [3][V][V]
  float *dense;
  int dense_ld;
  unsigned int *dbg;
};

template <int IC, int V>
struct TcAttnCfg {
  static constexpr int kSkp = (V + 3) / 4 * 4;                 // skeleton pitch in the theta buffer == dense_vp
  static constexpr int kSkel = kTileRows / V;                  // skeletons per tile
  static constexpr int kThetaPitch = kSkel * kSkp;             // floats per channel row
  static constexpr int kBBytes = 4 * IC * kBK * 2;             // stacked hi + lo rows
  static constexpr int kStageBytes = 2 * kABytes + kBBytes;
  // two epilogue groups work on alternate items, each with its own theta / phi buffers; the widest embedding pays
  // for them with the second operand stage (its epilogue, not the mainloop, is what bounds the kernel)
  static constexpr int kStages = IC == 64 ? 1 : 2;
  static constexpr int kStageStride = 2 * kABytes + 4 * 64 * kBK * 2;  // sized for IC = 64: 1024-byte aligned
  static constexpr int kThetaOff = kStages * kStageStride;
  static constexpr int kPhiOff = kThetaOff + IC * kThetaPitch * 4;
  static constexpr int kGroupBytes = IC * kThetaPitch * 4 + IC * kTileRows * 4;  // theta + phi of one group
  static constexpr int kAdjOff = kThetaOff + 2 * kGroupBytes;
  static constexpr int kBiasOff = kAdjOff + (3 * V * V * 4 + 15) / 16 * 16;
  static constexpr int kBarOff = kBiasOff + 6 * IC * 4;
  static constexpr int kSmemBytes = kBarOff + 128 + 1024;
  static constexpr int kAccCols = 4 * IC;                      // hi-product half | lo-weight half
  static constexpr int kTmemCols = 2 * kAccCols < 32 ? 32 : 2 * kAccCols;
  static_assert(kSmemBytes <= kSmemLimit, "shared memory budget");
  static_assert(IC % 16 == 0 && IC <= 64, "embedding width");
};

// One token row w of the attention (thread = row): S[v] = <theta[v], phi[w]> / IC over the V vertices of the row's
// skeleton, softmax over v, plus the static term; written as the row's mixing coefficients of partition `part`.
// theta_s: [IC][kThetaPitch] skeleton-padded, phi_s: [IC][128], adj_s: [3][V][V].
template <int IC, int V>
__device__ __forceinline__ void attn_softmax_row(const float *theta_s, const float *phi_s, const float *adj_s, int part, int row,
                                                 int th_col, int wv, float *dense_row) {
  constexpr int kSkp = (V + 3) / 4 * 4;
  constexpr int kThetaPitch = (kTileRows / V) * kSkp;
  float sv[kSkp];
#pragma unroll
  for (int v = 0; v < kSkp; ++v) sv[v] = 0.f;
#pragma unroll 2
  for (int c = 0; c < IC; ++c) {
    const float ph = phi_s[c * kTileRows + row];
    const float4 *th = reinterpret_cast<const float4 *>(theta_s + c * kThetaPitch + th_col);
#pragma unroll
    for (int j = 0; j < kSkp / 4; ++j) {
      const float4 t = th[j];
      sv[4 * j] = fmaf(t.x, ph, sv[4 * j]);
      sv[4 * j + 1] = fmaf(t.y, ph, sv[4 * j + 1]);
      sv[4 * j + 2] = fmaf(t.z, ph, sv[4 * j + 2]);
      sv[4 * j + 3] = fmaf(t.w, ph, sv[4 * j + 3]);
    }
  }
  float mx = -INFINITY;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    sv[v] = sv[v] / (float)IC;
    mx = fmaxf(mx, sv[v]);
  }
  float sum = 0.f;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    sv[v] = expf(sv[v] - mx);
    sum += sv[v];
  }
  const float inv = 1.0f / sum;
#pragma unroll
  for (int v = 0; v < kSkp; ++v) sv[v] = v < V ? fmaf(sv[v], inv, adj_s[(part * V + v) * V + wv]) : 0.f;
  float4 *dst = reinterpret_cast<float4 *>(dense_row + part * kSkp);
#pragma unroll
  for (int j = 0; j < kSkp / 4; ++j) dst[j] = make_float4(sv[4 * j], sv[4 * j + 1], sv[4 * j + 2], sv[4 * j + 3]);
}

template <int IC, int V>
__global__ void __launch_bounds__(384, 1) k_tc_attn(const __grid_constant__ TcAttnArgs a) {
  using Cfg = TcAttnCfg<IC, V>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  float *adj_s = reinterpret_cast<float *>(smem + Cfg::kAdjOff);      // [3][V][V]
  float *bias_s = reinterpret_cast<float *>(smem + Cfg::kBiasOff);    // [3][2*IC]
  uint64_t *full = reinterpret_cast<uint64_t *>(smem + Cfg::kBarOff);
  uint64_t *empty = full + Cfg::kStages;
  uint64_t *tfull = empty + Cfg::kStages;
  uint64_t *tempty = tfull + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + 2);
  const uint32_t smem_base = ptx::smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cta = blockIdx.x, ncta = gridDim.x;
  pdl_trigger();
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], 4);
    }
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&a.tm_x);
    ptx::prefetch_tmap(&a.tm_w);
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish();
  }
  for (int i = threadIdx.x; i < 3 * V * V; i += blockDim.x) adj_s[i] = a.adj[i];
  for (int i = threadIdx.x; i < 6 * IC; i += blockDim.x) bias_s[i] = a.bias[i];
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  const int nkb = a.cin / kBK;

  if (warp == 0) {
    if (lane == 0) {
      PipeState ps;
      bool ok = true;
      for (int tile = cta; ok && tile < a.n_tiles; tile += ncta) {
        const int row = a.x_row + tile * a.tile_tokens;
        for (int part = 0; ok && part < 3; ++part) {
          for (int kc = 0; kc < nkb; ++kc) {
            ok = ptx::mbar_wait(&empty[ps.stage], ps.phase ^ 1, a.dbg, kDbgProdEmpty | (unsigned)(part * 16 + kc));
            if (!ok) break;
            const uint32_t st = smem_base + ps.stage * Cfg::kStageStride;
            ptx::mbar_arrive_expect_tx(&full[ps.stage], Cfg::kStageBytes);
            ptx::tma_load_2d_hint(st, &a.tm_x, &full[ps.stage], kc * kBK, row, ptx::kEvictNormal);
            ptx::tma_load_2d_hint(st + kABytes, &a.tm_x, &full[ps.stage], kc * kBK, row + a.t_alloc, ptx::kEvictNormal);
            ptx::tma_load_2d_hint(st + 2 * kABytes, &a.tm_w, &full[ps.stage], kc * kBK, part * 4 * IC, ptx::kEvictLast);
            ps.advance<Cfg::kStages>();
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      PipeState ps;
      bool ok = true;
      int it = 0;
      for (int tile = cta; ok && tile < a.n_tiles; tile += ncta) {
        for (int part = 0; ok && part < 3; ++part, ++it) {
          const int acc = it & 1;
          ok = ptx::mbar_wait(&tempty[acc], ((it >> 1) & 1) ^ 1, a.dbg, kDbgMmaTmemEmpty | (unsigned)it);
          if (!ok) break;
          ptx::tc_fence_after();
          const uint32_t d = tmem_base + acc * Cfg::kAccCols;
          for (int kc = 0; kc < nkb; ++kc) {
            ok = ptx::mbar_wait(&full[ps.stage], ps.phase, a.dbg, kDbgMmaFull | (unsigned)(part * 16 + kc));
            if (!ok) break;
            ptx::tc_fence_after();
            const uint32_t st = smem_base + ps.stage * Cfg::kStageStride;
            issue_kblock_stacked<4 * IC>(d, st, st + kABytes, st + 2 * kABytes, kc == 0);
            ptx::umma_commit(&empty[ps.stage]);
            ps.advance<Cfg::kStages>();
          }
          if (ok) ptx::umma_commit(&tfull[acc]);
        }
      }
    }
  } else if (warp >= 4) {
    // two groups of four warps (4..7, 8..11): group g owns accumulator g and takes the items with (it & 1) == g
    const int grp = (warp - 4) >> 2;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const bool row_ok = row < a.tile_tokens;
    const int sk = row_ok ? row / V : 0, wv = row_ok ? row - sk * V : 0;
    const int th_col = sk * Cfg::kSkp;  // this row's skeleton in the theta buffer
    float *theta_s = reinterpret_cast<float *>(smem + Cfg::kThetaOff + grp * Cfg::kGroupBytes);  // [IC][kThetaPitch]
    float *phi_s = reinterpret_cast<float *>(smem + Cfg::kPhiOff + grp * Cfg::kGroupBytes);      // [IC][128]
    bool ok = true;
    int it = 0;
    for (int tile = cta; tile < a.n_tiles; tile += ncta) {
      const long long tok = (long long)tile * a.tile_tokens + row;
      const bool valid = row_ok && tok < a.n_tokens;
      for (int part = 0; part < 3; ++part, ++it) {
        const int acc = it & 1;
        if (acc != grp) continue;
        // a warp whose wait expired keeps walking the items (named barriers below), it only stops computing
        if (ok) ok = ptx::mbar_wait(&tfull[acc], (it >> 1) & 1, a.dbg, kDbgEpiTmemFull | (unsigned)it);
        if (ok) {
          ptx::tc_fence_after();
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * Cfg::kAccCols;
#pragma unroll 1
          for (int c0 = 0; c0 < 2 * IC; c0 += 16) {
            uint32_t yh[16], yl[16];
            ptx::tmem_ld_32x16(taddr + c0, yh);
            ptx::tmem_ld_32x16(taddr + 2 * IC + c0, yl);
            ptx::tmem_ld_wait();
            if (row_ok) {
              const float *bb = bias_s + part * 2 * IC + c0;
              if (c0 < IC) {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                  theta_s[(c0 + j) * Cfg::kThetaPitch + th_col + wv] = __uint_as_float(yh[j]) + __uint_as_float(yl[j]) + bb[j];
              } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                  phi_s[(c0 - IC + j) * kTileRows + row] = __uint_as_float(yh[j]) + __uint_as_float(yl[j]) + bb[j];
              }
            }
          }
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&tempty[acc]);  // accumulator drained: the next item's MMAs may start
        }
        asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");  // theta / phi of the whole tile are in shared memory
        if (ok && valid) attn_softmax_row<IC, V>(theta_s, phi_s, adj_s, part, row, th_col, wv, a.dense + tok * a.dense_ld);
        asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");  // buffers free for the group's next item
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

// Attention half for a narrow input (cin <= 8: the 3-channel first layer): the embeddings are a handful of
// FMAs per token, so there is no GEMM to speak of -- each thread computes theta / phi of its token row straight
// into the shared-memory buffers and the same per-row softmax follows.  One token tile per CTA, 128 threads.
struct AttnSmallArgs {
  const __nv_bfloat16 *x_hi, *x_lo;
  int cs_in, cin;
  const float *w;     // [cin][6*IC] k-major
  const float *bias;  // [6*IC]
  const float *adj;
  long long n_tokens;
  int tile_tokens;
  float *dense;
  int dense_ld;
};

template <int IC, int V>
__global__ void __launch_bounds__(128) k_attn_small(AttnSmallArgs a) {
  constexpr int kSkp = (V + 3) / 4 * 4;
  constexpr int kThetaPitch = (kTileRows / V) * kSkp;
  __shared__ __align__(16) float theta_s[IC * kThetaPitch];
  __shared__ __align__(16) float phi_s[IC * kTileRows];
  __shared__ float adj_s[3 * V * V];
  __shared__ float w_s[8 * 6 * IC + 6 * IC];
  pdl_trigger();
  for (int i = threadIdx.x; i < 3 * V * V; i += blockDim.x) adj_s[i] = a.adj[i];
  for (int i = threadIdx.x; i < a.cin * 6 * IC; i += blockDim.x) w_s[i] = a.w[i];
  for (int i = threadIdx.x; i < 6 * IC; i += blockDim.x) w_s[8 * 6 * IC + i] = a.bias[i];
  pdl_wait();
  const int row = threadIdx.x;
  const long long tok = (long long)blockIdx.x * a.tile_tokens + row;
  const bool valid = row < a.tile_tokens && tok < a.n_tokens;
  const int sk = row < a.tile_tokens ? row / V : 0, wv = row < a.tile_tokens ? row - sk * V : 0;
  const int th_col = sk * kSkp;
  float x[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) x[c] = (valid && c < a.cin) ? join_bf16(a.x_hi[tok * a.cs_in + c], a.x_lo[tok * a.cs_in + c]) : 0.f;
  __syncthreads();
  for (int part = 0; part < 3; ++part) {
    if (row < a.tile_tokens) {
#pragma unroll 4
      for (int n = 0; n < 2 * IC; ++n) {
        float v = w_s[8 * 6 * IC + part * 2 * IC + n];
#pragma unroll
        for (int c = 0; c < 8; ++c)
          if (c < a.cin) v = fmaf(x[c], w_s[c * 6 * IC + part * 2 * IC + n], v);
        if (n < IC) theta_s[n * kThetaPitch + th_col + wv] = v;
        else phi_s[(n - IC) * kTileRows + row] = v;
      }
    }
    __syncthreads();
    if (valid) attn_softmax_row<IC, V>(theta_s, phi_s, adj_s, part, row, th_col, wv, a.dense + tok * a.dense_ld);
    __syncthreads();
  }
}

// =============================================================================================
// Self-attention unit of CoS-TR, qkv conv + attention in one kernel (GcnUnitAttention / SpatialAttention with
// only_attention, models/s_tr/s_tr.py:134-231,417-476).  Work item = (token tile, group of G = 64/DVH heads): the
// mainloop computes the group's [q (16) | k (16) | v (64)] = 96 columns of the qkv conv on tcgen05 (stacked split
// products: the group's hi and lo weight rows are adjacent, one operand of 192 rows), on the data_bn-normalised input
// rows.  Two epilogue groups of four warps take alternate items (own TMEM accumulator and shared-memory buffers each;
// thread = token row): q stays in registers, k and v of the tile go to shared memory as fp32, then per head
// w_j = softmax_j <q_i, k_j> over the V vertices of the row's skeleton and out_i = sum_j w_j v_j, written as packed
// split-bf16 rows -- the operand of the unit's output conv.  q, k, v never travel through memory.
// =============================================================================================
struct TcSaArgs {
  CUtensorMap tm_x;  // normalised input rows (1 slot), box {64, 128}
  CUtensorMap tm_w;  // [items][hi: q, k, v of the group | lo: same][cin], box {64, 192}
  int x_row, t_alloc, cin;
  int n_tiles, tile_tokens, V;
  long long n_tokens;
  const float *bias;  // [items][96]
  __nv_bfloat16 *y_hi, *y_lo;
  int cs_out;
  unsigned int *dbg;
};

template <int DVH>
struct TcSaCfg {
  static constexpr int kDkh = DVH / 4;
  static constexpr int kHeadsPerItem = 64 / DVH;  // 8, 4, 2
  static constexpr int kItems = 8 / kHeadsPerItem;  // per tile: 1, 2, 4
  static constexpr int kN = 96;                   // q 16 | k 16 | v 64
  static constexpr int kBBytes = 2 * kN * kBK * 2;  // stacked hi + lo rows: 24 KB
  static constexpr int kStageBytes = 2 * kABytes + kBBytes;
  static constexpr int kStageStride = (kStageBytes + 1023) / 1024 * 1024;
  static constexpr int kStages = 2;
  static constexpr int kVPitch = 64 + 4;
  static constexpr int kGroupBytes = kTileRows * 16 * 4 + kTileRows * kVPitch * 4;  // k + v of one epilogue group
  static constexpr int kKOff = kStages * kStageStride;
  static constexpr int kBiasOff = kKOff + 2 * kGroupBytes;
  static constexpr int kBarOff = kBiasOff + 4 * kN * 4;
  static constexpr int kSmemBytes = kBarOff + 128 + 1024;
  static constexpr int kAccStride = 256;
  static constexpr int kTmemCols = 512;
  static_assert(kSmemBytes <= kSmemLimit, "shared memory budget");
};

template <int DVH>
__global__ void __launch_bounds__(384, 1) k_tc_sa(const __grid_constant__ TcSaArgs a) {
  using Cfg = TcSaCfg<DVH>;
  constexpr int DKH = Cfg::kDkh, G = Cfg::kHeadsPerItem, NI = Cfg::kItems, N = Cfg::kN;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  float *bias_s = reinterpret_cast<float *>(smem + Cfg::kBiasOff);  // [NI][96]
  uint64_t *full = reinterpret_cast<uint64_t *>(smem + Cfg::kBarOff);
  uint64_t *empty = full + Cfg::kStages;
  uint64_t *tfull = empty + Cfg::kStages;
  uint64_t *tempty = tfull + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + 2);
  const uint32_t smem_base = ptx::smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cta = blockIdx.x, ncta = gridDim.x;
  pdl_trigger();
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], 4);
    }
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&a.tm_x);
    ptx::prefetch_tmap(&a.tm_w);
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish();
  }
  for (int i = threadIdx.x; i < NI * N; i += blockDim.x) bias_s[i] = a.bias[i];
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  const int nkb = a.cin / kBK;

  if (warp == 0) {
    if (lane == 0) {
      PipeState ps;
      bool ok = true;
      for (int tile = cta; ok && tile < a.n_tiles; tile += ncta) {
        const int row = a.x_row + tile * a.tile_tokens;
        for (int item = 0; ok && item < NI; ++item) {
          for (int kc = 0; kc < nkb; ++kc) {
            ok = ptx::mbar_wait(&empty[ps.stage], ps.phase ^ 1, a.dbg, kDbgProdEmpty | (unsigned)(item * 16 + kc));
            if (!ok) break;
            const uint32_t st = smem_base + ps.stage * Cfg::kStageStride;
            ptx::mbar_arrive_expect_tx(&full[ps.stage], Cfg::kStageBytes);
            ptx::tma_load_2d_hint(st, &a.tm_x, &full[ps.stage], kc * kBK, row, ptx::kEvictNormal);
            ptx::tma_load_2d_hint(st + kABytes, &a.tm_x, &full[ps.stage], kc * kBK, row + a.t_alloc, ptx::kEvictNormal);
            ptx::tma_load_2d_hint(st + 2 * kABytes, &a.tm_w, &full[ps.stage], kc * kBK, item * 2 * N, ptx::kEvictLast);
            ps.advance<Cfg::kStages>();
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      PipeState ps;
      bool ok = true;
      int it = 0;
      for (int tile = cta; ok && tile < a.n_tiles; tile += ncta) {
        for (int item = 0; ok && item < NI; ++item, ++it) {
          const int acc = it & 1;
          ok = ptx::mbar_wait(&tempty[acc], ((it >> 1) & 1) ^ 1, a.dbg, kDbgMmaTmemEmpty | (unsigned)it);
          if (!ok) break;
          ptx::tc_fence_after();
          const uint32_t d = tmem_base + acc * Cfg::kAccStride;
          for (int kc = 0; kc < nkb; ++kc) {
            ok = ptx::mbar_wait(&full[ps.stage], ps.phase, a.dbg, kDbgMmaFull | (unsigned)(item * 16 + kc));
            if (!ok) break;
            ptx::tc_fence_after();
            const uint32_t st = smem_base + ps.stage * Cfg::kStageStride;
            issue_kblock_stacked<2 * N>(d, st, st + kABytes, st + 2 * kABytes, kc == 0);
            ptx::umma_commit(&empty[ps.stage]);
            ps.advance<Cfg::kStages>();
          }
          if (ok) ptx::umma_commit(&tfull[acc]);
        }
      }
    }
  } else if (warp >= 4) {
    const int grp = (warp - 4) >> 2;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const bool row_ok = row < a.tile_tokens;
    const int sk0 = row_ok ? row - row % a.V : 0;
    float *k_s = reinterpret_cast<float *>(smem + Cfg::kKOff + grp * Cfg::kGroupBytes);  // [128][16]
    float *v_s = k_s + kTileRows * 16;                                                    // [128][kVPitch]
    bool ok = true;
    int it = 0;
    for (int tile = cta; tile < a.n_tiles; tile += ncta) {
      const long long tok = (long long)tile * a.tile_tokens + row;
      const bool valid = row_ok && tok < a.n_tokens;
      for (int item = 0; item < NI; ++item, ++it) {
        const int acc = it & 1;
        if (acc != grp) continue;
        float qv[16];
        if (ok) ok = ptx::mbar_wait(&tfull[acc], (it >> 1) & 1, a.dbg, kDbgEpiTmemFull | (unsigned)it);
        if (ok) {
          ptx::tc_fence_after();
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * Cfg::kAccStride;
          const float *bb = bias_s + item * N;
#pragma unroll 1
          for (int c0 = 0; c0 < N; c0 += 16) {
            uint32_t yh[16], yl[16];
            ptx::tmem_ld_32x16(taddr + c0, yh);
            ptx::tmem_ld_32x16(taddr + N + c0, yl);
            ptx::tmem_ld_wait();
            float x[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = __uint_as_float(yh[j]) + __uint_as_float(yl[j]) + bb[c0 + j];
            if (c0 == 0) {
#pragma unroll
              for (int j = 0; j < 16; ++j) qv[j] = x[j];
            } else if (c0 == 16) {
#pragma unroll
              for (int j4 = 0; j4 < 4; ++j4)
                *reinterpret_cast<float4 *>(k_s + row * 16 + 4 * j4) = make_float4(x[4 * j4], x[4 * j4 + 1], x[4 * j4 + 2], x[4 * j4 + 3]);
            } else {
#pragma unroll
              for (int j4 = 0; j4 < 4; ++j4)
                *reinterpret_cast<float4 *>(v_s + row * Cfg::kVPitch + (c0 - 32) + 4 * j4) =
                    make_float4(x[4 * j4], x[4 * j4 + 1], x[4 * j4 + 2], x[4 * j4 + 3]);
            }
          }
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&tempty[acc]);  // accumulator drained: the next item's MMAs may start
        }
        asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");  // k / v of the whole tile are in shared memory
        if (ok && valid) {
#pragma unroll
          for (int g = 0; g < G; ++g) {  // unrolled: q stays in registers
            float w[kAttnMaxV];
            float mx = -INFINITY;
#pragma unroll
            for (int j = 0; j < kAttnMaxV; ++j) {
              if (j < a.V) {
                float sdot = 0.f;
                if (DKH >= 4) {
#pragma unroll
                  for (int d4 = 0; d4 < DKH / 4; ++d4) {
                    const float4 k4 = *reinterpret_cast<const float4 *>(k_s + (sk0 + j) * 16 + g * DKH + 4 * d4);
                    sdot = fmaf(qv[g * DKH + 4 * d4], k4.x, sdot);
                    sdot = fmaf(qv[g * DKH + 4 * d4 + 1], k4.y, sdot);
                    sdot = fmaf(qv[g * DKH + 4 * d4 + 2], k4.z, sdot);
                    sdot = fmaf(qv[g * DKH + 4 * d4 + 3], k4.w, sdot);
                  }
                } else {
                  const float2 k2 = *reinterpret_cast<const float2 *>(k_s + (sk0 + j) * 16 + g * 2);
                  sdot = fmaf(qv[g * 2], k2.x, qv[g * 2 + 1] * k2.y);
                }
                w[j] = sdot;
                mx = fmaxf(mx, sdot);
              } else {
                w[j] = 0.f;
              }
            }
            float sum = 0.f;
#pragma unroll
            for (int j = 0; j < kAttnMaxV; ++j)
              if (j < a.V) {
                w[j] = expf(w[j] - mx);
                sum += w[j];
              }
            const float inv = 1.0f / sum;
            float o[DVH];
#pragma unroll
            for (int d = 0; d < DVH; ++d) o[d] = 0.f;
#pragma unroll
            for (int j = 0; j < kAttnMaxV; ++j)
              if (j < a.V) {
                const float wj = w[j] * inv;
#pragma unroll
                for (int d4 = 0; d4 < DVH / 4; ++d4) {
                  const float4 v4 = *reinterpret_cast<const float4 *>(v_s + (sk0 + j) * Cfg::kVPitch + g * DVH + 4 * d4);
                  o[4 * d4] = fmaf(wj, v4.x, o[4 * d4]);
                  o[4 * d4 + 1] = fmaf(wj, v4.y, o[4 * d4 + 1]);
                  o[4 * d4 + 2] = fmaf(wj, v4.z, o[4 * d4 + 2]);
                  o[4 * d4 + 3] = fmaf(wj, v4.w, o[4 * d4 + 3]);
                }
              }
            const int col = (item * G + g) * DVH;
#pragma unroll
            for (int e = 0; e < DVH / 8; ++e) {
              uint32_t oh[4], ol[4];
#pragma unroll
              for (int w2 = 0; w2 < 4; ++w2) {
                const float x0 = o[8 * e + 2 * w2], x1 = o[8 * e + 2 * w2 + 1];
                oh[w2] = pack_bf16x2(x0, x1);
                ol[w2] = pack_bf16x2(x0 - bf16_lo_as_float(oh[w2]), x1 - bf16_hi_as_float(oh[w2]));
              }
              *reinterpret_cast<uint4 *>(a.y_hi + tok * a.cs_out + col + 8 * e) = make_uint4(oh[0], oh[1], oh[2], oh[3]);
              *reinterpret_cast<uint4 *>(a.y_lo + tok * a.cs_out + col + 8 * e) = make_uint4(ol[0], ol[1], ol[2], ol[3]);
            }
          }
        }
        asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");  // buffers free for the group's next item
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

}  // namespace cosk
