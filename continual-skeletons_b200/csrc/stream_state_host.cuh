// Host half of the per-stream state calls (cosk_reset_streams, cosk_export_streams, cosk_import_streams,
// cosk_resize_batch, cosk_prime_streams): the payload layout of a batch as a StateArgs table, index checks, and the one
// k_stream_state launch per call on the batch it is handed.
// Part of cosk.cu (included after its helpers, whose names it uses); the kernel is in stream_state.cuh.  The step route
// table of the GPU tests covers the step kernels; k_stream_state is checked by tests/test_gpu_streams.py.
#pragma once

namespace {

// ---- per-stream state (k_stream_state) -------------------------------------------------------------------------------
// The payload of a stream, in this order: the input ring, then per block its temporal ring and its output ring, then the
// pooling window and its sum (models with a head).  Each ring holds only the entries a later step can read, newest first,
// each entry as its planes (hi, lo for the bf16 rings):
//   input ring        kResDelay entries if block 0 has a residual (x_{n-4}), else none
//   temporal ring     the kTaps - 1 history taps
//   output ring       kResDelay entries if the next block has a residual, else the newest (cosk_read_block); the head
//                     and the next block consume the newest within the step that produced it
//   pooling window    all pool_size entries (fp32 [c_last]), then the fp64 running sum [c_last]
// Entry e of a ring whose counter (entries written so far) is cnt sits in slot (cnt - 1 - e) mod slots: the slot
// arithmetic of the step (RingWalk, n mod R), so the payload does not depend on the time chunk, N or tile position.
// The stride-2 blocks read two of their four input entries; all four are kept so the layout has no phase.
void add_ring(StateArgs &a, long long &off, void *base, long long plane_bytes, int run_bytes, int planes, int entries, int slots,
              long long cnt) {
  if (entries == 0) return;
  StateRing &r = a.ring[a.n_rings];
  r.payload_off = off;
  r.run_bytes = run_bytes;
  r.planes = planes;
  r.entries = entries;
  r.slots = slots;
  r.newest = mod_slot(cnt - 1, slots);
  r.first_run = a.runs;
  a.state[a.n_rings] = {static_cast<char *>(base), plane_bytes};
  a.n_rings++;
  a.runs += entries * planes;
  off += (long long)entries * planes * run_bytes;
}

void add_act_ring(const cosk_model *m, StateArgs &a, long long &off, const ActBuf &b, int c, int slots, int entries, long long cnt) {
  const int cs = round_up(c, 8);
  const int run = m->cfg.persons * m->cfg.vertices * cs * (int)sizeof(__nv_bfloat16);
  add_ring(a, off, b.ptr, (long long)b.t_alloc * cs * (long long)sizeof(__nv_bfloat16), run, 2, entries, slots, cnt);
}

// The layout above for the buffers and counters of a batch (an empty batch: geometry only).
StateArgs state_args(const cosk_model *m, const Batch &bt) {
  const cosk_config &c = m->cfg;
  StateArgs a;
  memset(&a, 0, sizeof a);
  long long off = 0;
  const int first_res = c.blocks[0].res_kind != COSK_RES_NONE ? kResDelay : 0;
  add_act_ring(m, a, off, bt.xin, c.c_in, bt.Ro, first_res, bt.cnt.n_in[0]);
  for (int i = 0; i < c.n_blocks; ++i) {
    const bool next_res = i + 1 < c.n_blocks && c.blocks[i + 1].res_kind != COSK_RES_NONE;
    add_act_ring(m, a, off, bt.blk[i].ring, c.blocks[i].cout, bt.R, kTaps - 1, bt.cnt.n_in[i]);
    add_act_ring(m, a, off, bt.blk[i].out, c.blocks[i].cout, bt.Ro, next_res ? kResDelay : 1, bt.cnt.n_out[i]);
  }
  if (c.classes > 0) {
    const int cl = c.blocks[c.n_blocks - 1].cout;
    add_ring(a, off, bt.d_pool_ring, bt.n_streams * cl * (long long)sizeof(float), cl * (int)sizeof(float), 1, c.pool_size,
             c.pool_size, bt.cnt.pool_n);
    add_ring(a, off, bt.d_pool_sum, bt.n_streams * cl * (long long)sizeof(double), cl * (int)sizeof(double), 1, 1, 1, 1);
  }
  a.stream_bytes = off;
  return a;
}

// Host index list -> bounds and distinctness checked copy in m->h_idx.  lo = -1 admits "no source".
int check_indices(cosk_model *m, const int64_t *idx, int64_t n, long long lo, long long hi, bool distinct) {
  if (n < 0 || (n > 0 && !idx)) return fail(m, COSK_ERR_ARG, "bad index list");
  if (n > hi && distinct) return fail(m, COSK_ERR_ARG, "%lld indices for %lld streams", (long long)n, hi);
  std::vector<char> seen(distinct ? (size_t)hi : 0, 0);
  for (int64_t q = 0; q < n; ++q) {
    if (idx[q] < lo || idx[q] >= hi) return fail(m, COSK_ERR_ARG, "stream index %lld out of range [%lld, %lld)", (long long)idx[q], lo, hi);
    if (distinct && idx[q] >= 0 && seen[(size_t)idx[q]]++) return fail(m, COSK_ERR_ARG, "stream index %lld repeats", (long long)idx[q]);
  }
  m->h_idx.assign(idx, idx + n);
  return COSK_OK;
}

// One k_stream_state launch over the m->h_idx streams of batch `bt` (kStateMove: from the batch `from`).  The index upload
// waits for the previous call's kernel, which may read the same device buffer, so calls on different CUDA streams cannot
// overwrite each other's indices.
int launch_stream_state(cosk_model *m, const Batch &bt, int mode, void *payload, cudaStream_t s, const Batch *from = nullptr) {
  const long long k = (long long)m->h_idx.size();
  if (k == 0) return COSK_OK;
  if (!m->ev_idx) CK(cudaEventCreateWithFlags(&m->ev_idx, cudaEventDisableTiming));
  else CK(cudaStreamWaitEvent(s, m->ev_idx, 0));
  CK(cudaMemcpyAsync(bt.d_idx, m->h_idx.data(), (size_t)k * sizeof(long long), cudaMemcpyHostToDevice, s));
  StateArgs a = state_args(m, bt);
  if (from) memcpy(a.from, state_args(m, *from).state, sizeof a.from);
  a.mode = mode;
  a.k = k;
  a.idx = bt.d_idx;
  a.payload = static_cast<char *>(payload);
  const long long items = k * a.runs;
  const int grid = (int)std::min<long long>(items, (long long)m->num_sms * 8);
  CK(launch_k(k_stream_state, dim3(grid), dim3(256), 0, s, a));
  m->launches++;
  CK(cudaEventRecord(m->ev_idx, s));
  return COSK_OK;
}

// Fingerprint of every config field that shapes the payload or the meaning of its entries (FNV-1a).
uint64_t geometry_of(const cosk_config &c) {
  uint64_t h = 1469598103934665603ull;
  auto mix = [&](long long v) {
    for (int b = 0; b < 8; ++b) {
      h ^= (uint64_t)((v >> (8 * b)) & 0xff);
      h *= 1099511628211ull;
    }
  };
  mix(c.vertices), mix(c.persons), mix(c.c_in), mix(c.n_blocks), mix(c.padding);
  mix(c.classes > 0), mix(c.classes > 0 ? c.pool_size : 0), mix(c.classes > 0 ? c.pool_padding : 0);
  for (int i = 0; i < c.n_blocks; ++i) {
    const cosk_block_cfg &b = c.blocks[i];
    mix(b.cin), mix(b.cout), mix(b.stride), mix(b.res_kind), mix(b.gconv);
  }
  return h;
}

}  // namespace
