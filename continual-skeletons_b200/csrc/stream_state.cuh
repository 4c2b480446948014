// k_stream_state: the per-stream state of chosen streams -- zeroed, gathered into a payload, scattered from one, or moved
// into the buffers of another batch size -- in one launch.
//
// Which per-handle buffers are state (read by a later step) and which are scratch of the frame in flight:
//   state    xin             input ring: block 0 reads x_{n-4} of it as the delayed residual
//            blk[i].ring     temporal ring: the 8 history taps of the 9-tap conv
//            blk[i].out      block-output ring: x_{n-4} for the next block's residual; the newest entry is what
//                            cosk_read_block returns
//            d_pool_ring     pooling window [P][N][c_last] fp32, d_pool_sum its fp64 running sum [N][c_last]
//   scratch  blk[i].sa       attention rows of the frame in flight, written and read within one block step
//            blk[i].sa_x     the unit's data_bn-normalised input of the frame in flight
//            blk[i].sa_q     q | k | v rows of the frame in flight (unfused tensor-core qkv conv)
//            d_qkv           q | k | v rows of the frame in flight (SIMT attention)
//            d_dense         per-token mixing rows of the adaptive graph conv of the frame in flight
// Scratch is rewritten before it is read on every step and takes no part here.
//
// A stream's rows are contiguous in every plane of every state buffer: token (n*S + s)*V + v of a token-major ring
// (stream n owns S*V*cs bf16 of each plane, cs a multiple of 8, so 16-byte aligned runs), row n of the pooling
// buffers.  A "run" is one stream's rows of one (buffer, entry, plane); it is the unit of work, so the rows of a
// neighbour -- in the same token tile or not -- are never touched.
#pragma once
#include "common.cuh"

namespace cosk {

constexpr int kMaxStateRings = 2 * 16 + 3;  // input ring, temporal + output ring per block (COSK_MAX_BLOCKS), pool ring, pool sum

// Geometry of one state buffer, the same for every batch size.  Entry e (0 = newest) lives in slot (newest - e) mod slots;
// the payload stores entries in that order, each as `planes` runs of run_bytes.
struct StateRing {
  long long payload_off;  // bytes into a stream's payload
  int run_bytes, planes, entries, slots, newest;
  int first_run;  // runs of the rings before this one
};
// Where a buffer lives for one batch size: stream n's run of (slot, plane) starts at base + (slot*planes + plane)*plane_bytes
// + n*run_bytes.
struct StateSide {
  char *base;
  long long plane_bytes;
};

enum StateMode : int {
  kStateZero = 0,     // state of stream idx[q] := 0
  kStateGather = 1,   // payload row q := state of stream idx[q]
  kStateScatter = 2,  // state of stream idx[q] := payload row q
  kStateMove = 3,     // state of stream q := state of stream idx[q] in `from` (idx[q] < 0: zero)
};

struct StateArgs {
  StateRing ring[kMaxStateRings];
  StateSide state[kMaxStateRings];  // the handle's buffers
  StateSide from[kMaxStateRings];   // kStateMove: the buffers of the old batch size
  int n_rings, runs;                // runs = runs per stream
  int mode;
  long long k;                      // streams of the call
  const long long *idx;             // [k]
  char *payload;                    // [k][stream_bytes]
  long long stream_bytes;
};

__device__ __forceinline__ char *state_run(const StateSide &sd, const StateRing &r, int slot, int plane, long long n) {
  return sd.base + ((long long)slot * r.planes + plane) * sd.plane_bytes + n * r.run_bytes;
}

// Work item = one run of one stream; persistent CTAs stride over the k * runs items, the threads of a CTA over the
// 16-byte words of a run (4-byte words when a run is not 16-byte aligned: fp32 / fp64 pooling rows of c_last % 4 != 0).
__global__ void __launch_bounds__(256) k_stream_state(const __grid_constant__ StateArgs a) {
  pdl_trigger();
  pdl_wait();  // every state access below is ordered after the previous kernel on the stream
  const long long items = a.k * a.runs;
  for (long long it = blockIdx.x; it < items; it += gridDim.x) {
    const long long q = it / a.runs;
    const int run = (int)(it - q * a.runs);
    int g = 0;
    while (g + 1 < a.n_rings && a.ring[g + 1].first_run <= run) ++g;
    const StateRing &r = a.ring[g];
    const int e = (run - r.first_run) / r.planes, p = (run - r.first_run) % r.planes;
    const int slot = (r.newest - e + r.slots) % r.slots;
    const long long n = a.idx[q];
    const char *src = nullptr;
    char *dst;
    char *prow = a.payload + q * a.stream_bytes + r.payload_off + ((long long)e * r.planes + p) * r.run_bytes;
    switch (a.mode) {
      case kStateZero: dst = state_run(a.state[g], r, slot, p, n); break;
      case kStateGather: src = state_run(a.state[g], r, slot, p, n); dst = prow; break;
      case kStateScatter: src = prow; dst = state_run(a.state[g], r, slot, p, n); break;
      default:
        src = n >= 0 ? state_run(a.from[g], r, slot, p, n) : nullptr;
        dst = state_run(a.state[g], r, slot, p, q);
    }
    const bool v16 = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst) | (uintptr_t)r.run_bytes) & 15) == 0;
    if (v16) {
      // four loads in flight per thread before the first store (src and dst may alias as far as the compiler knows)
      constexpr int kBatch = 4;
      const int words = r.run_bytes >> 4;
      for (int w0 = threadIdx.x; w0 < words; w0 += kBatch * blockDim.x) {
        uint4 v[kBatch];
#pragma unroll
        for (int j = 0; j < kBatch; ++j) {
          const int w = w0 + j * blockDim.x;
          v[j] = src && w < words ? __ldg(reinterpret_cast<const uint4 *>(src) + w) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int j = 0; j < kBatch; ++j) {
          const int w = w0 + j * blockDim.x;
          if (w < words) reinterpret_cast<uint4 *>(dst)[w] = v[j];
        }
      }
    } else {
      const int words = r.run_bytes >> 2;
      for (int w = threadIdx.x; w < words; w += blockDim.x)
        reinterpret_cast<uint32_t *>(dst)[w] = src ? __ldg(reinterpret_cast<const uint32_t *>(src) + w) : 0u;
    }
  }
}

}  // namespace cosk
