// Graph conv with the channels on the TMEM lanes (k_tc_gcnt): GraphConvolution.forward, models/base.py:260-270.
//
//   z[:, w] = sum_i sum_v A_i[v, w] * (W_i x[:, v]) + R x[:, w] + bias ,  ReLU
//
// The token-major kernel (k_tc_gcn) computes Y = X W^T with token rows on the accumulator lanes, so the adjacency
// contraction runs ACROSS lanes: every accumulator column travels TMEM -> registers -> shared memory -> registers
// (drain and mix warps), and that epilogue -- not the tensor pipe, not HBM -- bounds the kernel.
//
// Here the GEMM is issued the other way round,  Y_i^T = W_i X^T :  the 128 output channels of a chunk are the UMMA M
// dimension (TMEM lanes), the tokens of TWO adjacent tiles are the N dimension (256 accumulator columns), operands are the
// very same K-major shared-memory tiles with the A and B roles swapped.  A thread of the epilogue then owns ONE output
// channel and sees all the tokens of its tile along the columns, skeleton after skeleton (V consecutive columns), so the
// adjacency contraction becomes register arithmetic inside the thread:
//
//   z[w]  = d0[w] * Y_0[w] + bias                      self links      (partition 0 is diagonal)
//   z[w] += c1[w] * Y_1[parent(w)]                     inward links    (every vertex has one parent in the skeleton tree)
//   z[p] += c2[a] * Y_2[a]  for every child a of p     outward links
//   z[w] += Y_3[w]                                     gcn_residual    (folded 1x1 conv or identity; folded into W_0 when d0 == 1)
//
// with the tree (which register feeds which) known at compile time -- the two skeletons the reference ships,
// datasets/ntu_rgbd.py:3-35 and datasets/kinetics.py:24-46 -- and the coefficients A * graph_attn read from the kernel
// parameters (constant bank operands of the FMAs).  No shared-memory exchange, no cross-lane traffic: ~3 FMAs per output.
// The host only selects this kernel when the block's mixing matrix has exactly this sparsity pattern (cosk.cu:prepare);
// anything else stays on k_tc_gcn.
//
// Work item = (frame, pair of adjacent token tiles); per item the X tiles stay resident in shared memory while the weight
// slabs of every (128-channel chunk, partition) stream through a 3-stage ring; one accumulator of 256 columns per
// (chunk, partition), double buffered in TMEM, consumed partition by partition while the next one is being computed.
//   warp 0  TMA producer (weights)   warp 2  TMA producer (X)   warp 1  MMA issuer + TMEM owner   warps 4-11  epilogue (group 0: tile a, group 1: tile b)
// The epilogue threads hold a whole tile row of outputs (125 fp32) in registers: the first warpgroup (producer, issuer, two
// idle warps) gives registers back with setmaxnreg and the two epilogue warpgroups take them (the CTA owns 384 * 168 registers: 128 * 56 + 256 * 224 after the trade).
#pragma once
#include <type_traits>
#include <utility>

#include "tc_kernels.cuh"

namespace cosk {

enum : unsigned int {
  kDbgGcntXEmpty = 0x31000000u,
  kDbgGcntWEmpty = 0x32000000u,
  kDbgGcntXFull = 0x33000000u,
  kDbgGcntWFull = 0x34000000u,
  kDbgGcntTEmpty = 0x35000000u,
  kDbgGcntTFull = 0x36000000u,
};

// parent of every vertex in the skeleton tree (-1: the root), 0-based
template <int V>
__host__ __device__ constexpr int skel_parent(int w);
template <>
__host__ __device__ constexpr int skel_parent<25>(int w) {  // NTU RGB+D: joint -> the joint it points to (toward joint 21)
  constexpr int p[25] = {1, 20, 20, 2, 20, 4, 5, 6, 20, 8, 9, 10, 0, 12, 13, 14, 0, 16, 17, 18, -1, 22, 7, 24, 11};
  return p[w];
}
template <>
__host__ __device__ constexpr int skel_parent<18>(int w) {  // OpenPose-18 (Kinetics-skeleton), toward joint 1
  constexpr int p[18] = {1, -1, 1, 2, 3, 1, 5, 6, 2, 8, 9, 5, 11, 12, 0, 0, 14, 15};
  return p[w];
}

// f(integral_constant<int, 0>) ... f(integral_constant<int, N-1>): loop indices that are constant expressions, so that the
// skeleton tree resolves to fixed registers
template <int... I, class F>
__device__ __forceinline__ void static_for_impl(std::integer_sequence<int, I...>, F &&f) {
  (f(std::integral_constant<int, I>{}), ...);
}
template <int N, class F>
__device__ __forceinline__ void static_for(F &&f) {
  static_for_impl(std::make_integer_sequence<int, N>{}, f);
}

// An item's GEMM steps in issue order: pass by pass (pass = (chunk, partition), one accumulator), K-block by K-block.
// (Advancing the last two passes together, so that X K-block 0 is released two steps before the item ends instead of one,
// was measured and did not pay: 0.071 vs 0.067 ms for the 128 -> 128 layer.)
struct GcntStep {
  int pass, kb;
};
template <int NKB>
__device__ __forceinline__ GcntStep gcnt_step(int j, int) {
  return {j / NKB, j % NKB};
}

struct TcGcntArgs {
  TcGcnArgs g;        // tm_w: weights [2 planes][chunk][part][128 channels] x cin, box {64, 128}
  float coef[3][32];  // d0[w], c1[w] (from the parent of w), c2[a] (child a into its parent)
  int n_parts;        // 3 (gcn_residual folded into W_0) or 4
};

template <int V, int NKB>
struct TcGcntCfg {
  static constexpr int kSkel = kTileRows / V;          // skeletons per tile
  static constexpr int kXSlotBytes = 4 * kABytes;      // one K-block of both tiles: [hi a | hi b | lo a | lo b]
  static constexpr int kXSlots = 2;
  static constexpr int kWStageBytes = 2 * kABytes;     // 128 channels x 64 K: hi, lo
  static constexpr int kWStages = 3;
  static constexpr int kXOff = 0;
  static constexpr int kWOff = kXSlots * kXSlotBytes;
  static constexpr int kBarOff = kWOff + kWStages * kWStageBytes;
  static constexpr int kSmemBytes = kBarOff + 256 + 1024;
  static constexpr int kAccCols = 256;
  static constexpr int kTmemCols = 512;
  static constexpr int kThreads = 384;
  static_assert(NKB <= kXSlots, "an item's K-blocks must fit the X ring");
  static_assert(kSmemBytes <= kSmemLimit, "shared memory budget");
};

__device__ __forceinline__ void st_bf16(__nv_bfloat16 *p, __nv_bfloat16 v) {
  asm volatile("st.global.L1::no_allocate.b16 [%0], %1;" ::"l"(p), "h"(*reinterpret_cast<const unsigned short *>(&v)) : "memory");
}

template <int V, int NKB, int COUT>
__global__ void __launch_bounds__(384, 1) k_tc_gcnt(const __grid_constant__ TcGcntArgs ta) {
  using Cfg = TcGcntCfg<V, NKB>;
  constexpr int S = Cfg::kSkel;
  constexpr int NZ = S * V;
  constexpr int kChunks = COUT / 128;
  const TcGcnArgs &a = ta.g;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *xfull = reinterpret_cast<uint64_t *>(smem + Cfg::kBarOff);
  uint64_t *xempty = xfull + Cfg::kXSlots;
  uint64_t *wfull = xempty + Cfg::kXSlots;
  uint64_t *wempty = wfull + Cfg::kWStages;
  uint64_t *tfull = wempty + Cfg::kWStages;
  uint64_t *tempty = tfull + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + 2);
  // phase timers (COSK_TRACE=1) live in shared memory so that they cost no registers: [0..4] epilogue warp 4 {wait acc, load + mix,
  // store, total, items}, [8..11] MMA issuer {wait acc free, wait X, wait W, total}, [12..13] producer {wait X free, wait W free}
  unsigned long long *trs = reinterpret_cast<unsigned long long *>(smem + Cfg::kBarOff + 128);
  const uint32_t smem_base = ptx::smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cta = (int)blockIdx.x, ncta = (int)gridDim.x;

  pdl_trigger();
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kXSlots; ++s) {
      ptx::mbar_init(&xfull[s], 1);
      ptx::mbar_init(&xempty[s], 1);
    }
    for (int s = 0; s < Cfg::kWStages; ++s) {
      ptx::mbar_init(&wfull[s], 1);
      ptx::mbar_init(&wempty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], 8);  // the eight epilogue warps
    }
    for (int i = 0; i < 16; ++i) trs[i] = 0;
    ptx::fence_barrier_init();
    ptx::prefetch_tmap(&a.tm_x);
    ptx::prefetch_tmap(&a.tm_w);
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();  // prologue above touched only static data; activations of the previous kernel from here on

  const int P = ta.n_parts;
  const int n_pass = kChunks * P, n_steps = n_pass * NKB;  // pass = (chunk, partition): one accumulator
  const int n_pairs = (a.n_tiles + 1) >> 1;
  const int n_items = n_pairs * a.n_frames;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
  if (warp == 0) {
    if (lane == 0) {
      // ---- TMA producer, weights: one slab per (item, chunk, partition, K-block), independent of the X stream below so
      // that the next item's first slabs are already in flight while its X tiles still wait for their slots ----------
      PipeState ws;
      bool ok = true;
      const bool tr = a.trace != nullptr && cta == 0;
      for (int vt = cta; ok && vt < n_items; vt += ncta)
        for (int j = 0; j < n_steps; ++j) {
          const GcntStep st = gcnt_step<NKB>(j, n_pass);
          const long long c1 = tr ? clock64() : 0;
          ok = ptx::mbar_wait(&wempty[ws.stage], ws.phase ^ 1, a.dbg, kDbgGcntWEmpty | (unsigned)(st.pass * 16 + st.kb));
          if (!ok) break;
          if (tr) trs[13] += clock64() - c1;
          const uint32_t wst = smem_base + Cfg::kWOff + ws.stage * Cfg::kWStageBytes;
          const int wrow = st.pass * 128;  // pass = chunk * P + part
          ptx::mbar_arrive_expect_tx(&wfull[ws.stage], Cfg::kWStageBytes);
          ptx::tma_load_2d_hint(wst, &a.tm_w, &wfull[ws.stage], st.kb * kBK, wrow, ptx::kEvictLast);
          ptx::tma_load_2d_hint(wst + kABytes, &a.tm_w, &wfull[ws.stage], st.kb * kBK, P * COUT + wrow, ptx::kEvictLast);
          ws.advance<Cfg::kWStages>();
        }
    }
  } else if (warp == 2) {
    if (lane == 0) {
      // ---- TMA producer, X: the K-blocks of both tiles once per item ---------------------------------------------------
      uint32_t xf = 0;  // X fills so far
      bool ok = true;
      const bool tr = a.trace != nullptr && cta == 0;
      for (int vt = cta; ok && vt < n_items; vt += ncta) {
        const int fr = vt / n_pairs, pair = vt - fr * n_pairs;
        const int row = gcn_x_row(a, fr) + 2 * pair * a.tile_tokens;
        for (int kb = 0; kb < NKB; ++kb, ++xf) {
          const uint32_t slot = xf & 1, use = xf >> 1;
          const long long c0 = tr ? clock64() : 0;
          ok = ptx::mbar_wait(&xempty[slot], (use & 1) ^ 1, a.dbg, kDbgGcntXEmpty | (xf & 0xffff));
          if (!ok) break;
          if (tr) trs[12] += clock64() - c0;
          const uint32_t xs = smem_base + Cfg::kXOff + slot * Cfg::kXSlotBytes;
          ptx::mbar_arrive_expect_tx(&xfull[slot], Cfg::kXSlotBytes);
          ptx::tma_load_2d_hint(xs, &a.tm_x, &xfull[slot], kb * kBK, row, ptx::kEvictFirst);
          ptx::tma_load_2d_hint(xs + kABytes, &a.tm_x, &xfull[slot], kb * kBK, row + a.tile_tokens, ptx::kEvictFirst);
          ptx::tma_load_2d_hint(xs + 2 * kABytes, &a.tm_x, &xfull[slot], kb * kBK, row + a.t_alloc, ptx::kEvictFirst);
          ptx::tma_load_2d_hint(xs + 3 * kABytes, &a.tm_x, &xfull[slot], kb * kBK, row + a.t_alloc + a.tile_tokens, ptx::kEvictFirst);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ---- MMA issuer: D[128 channels x 256 tokens] (+)= W_part[128 x 64] * X[256 x 64]^T, three split products ------
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(128, 256);
      PipeState ws;
      uint32_t pidx = 0, xf0 = 0;
      bool ok = true;
      const bool tr = a.trace != nullptr && cta == 0;
      if (tr) trs[11] = 0ull - (unsigned long long)clock64();
      for (int vt = cta; ok && vt < n_items; vt += ncta, xf0 += NKB, pidx += n_pass) {
        for (int j = 0; j < n_steps; ++j) {
          const GcntStep st = gcnt_step<NKB>(j, n_pass);
          const uint32_t pi = pidx + st.pass, buf = pi & 1;
          if (st.kb == 0) {  // first touch of this pass's accumulator
            const long long c0 = tr ? clock64() : 0;
            ok = ptx::mbar_wait(&tempty[buf], ((pi >> 1) & 1) ^ 1, a.dbg, kDbgGcntTEmpty | (pi & 0xffff));
            if (!ok) break;
            if (tr) trs[8] += clock64() - c0;
          }
          const uint32_t d = tmem_base + buf * Cfg::kAccCols;
          const uint32_t xf = xf0 + st.kb, slot = xf & 1;
          const long long c1 = tr ? clock64() : 0;
          ok = ptx::mbar_wait(&xfull[slot], (xf >> 1) & 1, a.dbg, kDbgGcntXFull | (xf & 0xffff));
          if (!ok) break;
          const long long c2 = tr ? clock64() : 0;
          ok = ptx::mbar_wait(&wfull[ws.stage], ws.phase, a.dbg, kDbgGcntWFull | (unsigned)(st.pass * 16 + st.kb));
          if (!ok) break;
          if (tr) {
            trs[9] += c2 - c1;
            trs[10] += clock64() - c2;
          }
          ptx::tc_fence_after();
          const uint32_t xs = smem_base + Cfg::kXOff + slot * Cfg::kXSlotBytes;
          const uint32_t wst = smem_base + Cfg::kWOff + ws.stage * Cfg::kWStageBytes;
          const uint32_t wh = ptx::umma_desc_lo(wst), wl = ptx::umma_desc_lo(wst + kABytes);
          const uint32_t xh = ptx::umma_desc_lo(xs), xl = ptx::umma_desc_lo(xs + 2 * kABytes);
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k) {
            ptx::umma_bf16_lo(d, wh + 2 * k, xh + 2 * k, idesc, (st.kb == 0 && k == 0) ? 0u : 1u);
            ptx::umma_bf16_lo(d, wl + 2 * k, xh + 2 * k, idesc, 1u);
            ptx::umma_bf16_lo(d, wh + 2 * k, xl + 2 * k, idesc, 1u);
          }
          ptx::umma_commit(&wempty[ws.stage]);
          if (st.pass == n_pass - 1) ptx::umma_commit(&xempty[slot]);  // the item's last reader of this K-block
          if (st.kb == NKB - 1) ptx::umma_commit(&tfull[buf]);
          ws.advance<Cfg::kWStages>();
        }
      }
      if (tr) trs[11] += clock64();
    }
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
    // ---- epilogue: thread = output channel, columns = the tokens of its group's tile ------------------------------------
    const int e = warp - 4, g = e >> 2, q = warp & 3;  // a warp reads the TMEM lanes of sub-partition warp % 4
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(g * 128);
    uint32_t pidx = 0;
    bool ok = true;
    const bool tr = a.trace != nullptr && cta == 0 && warp == 4 && lane == 0;
    if (tr) trs[3] = 0ull - (unsigned long long)clock64();
    const bool odd = (lane & 1) != 0;
    for (int vt = cta; ok && vt < n_items; vt += ncta) {
      const int fr = vt / n_pairs, pair = vt - fr * n_pairs;
      const int tile = 2 * pair + g;
      const long long tok0 = (long long)tile * a.tile_tokens;
      const EpiArgs epi = gcn_epi(a, fr);
      for (int chunk = 0; ok && chunk < kChunks; ++chunk) {
        const int ch = chunk * 128 + q * 32 + lane;
        const float bias = __ldg(epi.bias + ch);
        float z[NZ];
        // partition by partition, as the accumulators complete
        for (int part = 0; part < P; ++part, ++pidx) {
          const uint32_t buf = pidx & 1;
          const long long c0 = tr ? clock64() : 0;
          ok = ptx::mbar_wait(&tfull[buf], (pidx >> 1) & 1, a.dbg, kDbgGcntTFull | (pidx & 0xffff));
          if (!ok) break;
          const long long c1 = tr ? clock64() : 0;
          ptx::tc_fence_after();
          const uint32_t taddr = lane_base + buf * Cfg::kAccCols;
          static_for<S>([&](auto s_) {
            constexpr int s = decltype(s_)::value;
            constexpr int col0 = s * V < kTileRows - 32 ? s * V : kTileRows - 32;  // 32 columns from the skeleton's first token
            constexpr int off = s * V - col0;                                       // (clamped to stay inside the tile)
            uint32_t y[32];
            ptx::tmem_ld_32x32(taddr + col0, y);
            ptx::tmem_ld_wait();
            if (part == 0) {
              static_for<V>([&](auto w_) {
                constexpr int w = decltype(w_)::value;
                z[s * V + w] = fmaf(ta.coef[0][w], __uint_as_float(y[off + w]), bias);
              });
            } else if (part == 1) {
              static_for<V>([&](auto w_) {
                constexpr int w = decltype(w_)::value, p = skel_parent<V>(w);
                if constexpr (p >= 0) z[s * V + w] = fmaf(ta.coef[1][w], __uint_as_float(y[off + p]), z[s * V + w]);
              });
            } else if (part == 2) {
              static_for<V>([&](auto c_) {
                constexpr int c = decltype(c_)::value, p = skel_parent<V>(c);
                if constexpr (p >= 0) z[s * V + p] = fmaf(ta.coef[2][c], __uint_as_float(y[off + c]), z[s * V + p]);
              });
            } else {
              static_for<V>([&](auto w_) {
                constexpr int w = decltype(w_)::value;
                z[s * V + w] += __uint_as_float(y[off + w]);
              });
            }
          });
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&tempty[buf]);  // accumulator read: the MMA may overwrite it
          if (tr) {
            trs[0] += c1 - c0;
            trs[1] += clock64() - c1;
          }
        }
        if (!ok) break;
        const long long c2 = tr ? clock64() : 0;
        // ReLU, split, store: a warp writes 32 consecutive channels (64 bytes, two full sectors) per token and plane
        long long left = tile < a.n_tiles ? a.n_tokens - tok0 : 0;
        const int n_valid = left > NZ ? NZ : (left < 0 ? 0 : (int)left);  // tokens of this tile that exist
        if constexpr (NZ % 2 == 1) {  // odd token count: the last token on its own (stored first: in this order ptxas keeps
                                      // every z[] of k_tc_gcnt<25, 2, 256> in registers)
          if (NZ - 1 < n_valid) {
            const float x = fmaxf(z[NZ - 1], epi.floor);
            const __nv_bfloat16 h = __float2bfloat16_rn(x);
            st_bf16(epi.y_hi + (tok0 + NZ - 1) * COUT + ch, h);
            st_bf16(epi.y_lo + (tok0 + NZ - 1) * COUT + ch, __float2bfloat16_rn(x - __bfloat162float(h)));
          }
        }
        // lanes 2j and 2j+1 (channels c, c+1) trade: the even lane ends up with both channels of the even token, the odd lane
        // with both of the odd token -> one 32-bit store per plane and token pair instead of two 16-bit ones
        const uint32_t sel_keep = odd ? 0x7632u : 0x5410u, sel_send = odd ? 0x5410u : 0x7632u;
        const uint32_t sel_hi = odd ? 0x1054u : 0x5410u, sel_lo = odd ? 0x3276u : 0x7632u;
        __nv_bfloat16 *ph = epi.y_hi + (tok0 + (odd ? 1 : 0)) * COUT + (ch & ~1);
        __nv_bfloat16 *pl = epi.y_lo + (tok0 + (odd ? 1 : 0)) * COUT + (ch & ~1);
        static_for<NZ / 2>([&](auto t_) {
          constexpr int t = 2 * decltype(t_)::value;
          const float x0 = fmaxf(z[t], epi.floor), x1 = fmaxf(z[t + 1], epi.floor);
          const uint32_t h2 = pack_bf16x2(x0, x1);
          const uint32_t l2 = pack_bf16x2(x0 - bf16_lo_as_float(h2), x1 - bf16_hi_as_float(h2));
          const uint32_t keep = __byte_perm(h2, l2, sel_keep);  // (hi, lo) of this lane's token
          const uint32_t recv = __shfl_xor_sync(0xffffffffu, __byte_perm(h2, l2, sel_send), 1);
          if (t + (odd ? 1 : 0) < n_valid) {
            *reinterpret_cast<uint32_t *>(ph + t * COUT) = __byte_perm(keep, recv, sel_hi);
            *reinterpret_cast<uint32_t *>(pl + t * COUT) = __byte_perm(keep, recv, sel_lo);
          }
        });
        if (tr) {
          trs[2] += clock64() - c2;
          trs[4] += 1;
        }
      }
    }
    if (tr) trs[3] += clock64();
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
  if (a.trace != nullptr && cta == 0 && threadIdx.x < 16) a.trace[threadIdx.x] = trs[threadIdx.x];
}

}  // namespace cosk
