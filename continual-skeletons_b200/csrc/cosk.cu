// libcosk: C ABI + host-side step orchestration for the continual ST-GCN forward on sm_100a.
// See include/cosk.h for the contract and DESIGN.md for the data layout.
#include "../../include/cosk.h"

#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <string>
#include <utility>
#include <vector>

#include "simt_kernels.cuh"
#include "tc_kernels.cuh"
#include "tc_gcnt.cuh"
#ifdef COSK_WITH_AGCNT  // k_tc_agcnt has never run on hardware: compiled in only on request (lib.py: COSK_WITH_AGCNT=1)
#include "tc_agcnt.cuh"
#endif
#include "tc_block.cuh"
#include "stream_state.cuh"

using namespace cosk;

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

#ifdef COSK_WITH_AGCNT
constexpr bool kAgcntBuilt = true;
#else
constexpr bool kAgcntBuilt = false;
#endif

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
// q | k | v columns of the unfused tensor-core qkv conv (C = 64: 96 columns), padded to a temporal-conv kernel width
constexpr int kSaQkvCols = 128;
// ring slot of frame n (frames before the start of the stream, n < 0, map to slots that are still zero)
inline int mod_slot(long long n, int slots) { return (int)(((n % slots) + slots) % slots); }

struct ActBuf {  // token-major split-bf16 activation ring: [slots][plane hi/lo][t_alloc][cs]
  __nv_bfloat16 *ptr = nullptr;
  int slots = 0, cs = 0, c = 0;
  long long t_alloc = 0;
  bool has_map = false;
  CUtensorMap map;
  size_t bytes() const { return (size_t)slots * 2 * t_alloc * cs * sizeof(__nv_bfloat16); }
  __nv_bfloat16 *hi(int slot) const { return ptr + (size_t)slot * 2 * t_alloc * cs; }
  __nv_bfloat16 *lo(int slot) const { return hi(slot) + (size_t)t_alloc * cs; }
  long long row_hi(int slot) const { return (long long)slot * 2 * t_alloc; }
  long long slot_elems() const { return 2 * t_alloc * cs; }
};

// Which kernels serve a block.  prepare() decides it once per block; the launchers, the walk's batched_ok,
// cosk_describe and cosk_block_uses_tensor_cores only read it.
enum class GcnRoute : uint8_t {
  kSimt,       // k_gcn_simt
  kSmall,      // k_gcn_small: narrow first layer, weights and mixed inputs of a tile in shared memory
  kTc,         // k_tc_gcn<gcn_parts, 1 or 2 operand stages>: token-major GEMM, then the mix
  kTcT,        // k_tc_gcnt: channel-major, mix along the skeleton tree in registers
  kTcAgcn,     // adaptive graph conv: dense mix on k_tc_agcn
  kTcAgcnt,    // adaptive graph conv: dense mix on the channel-major k_tc_agcnt (COSK_WITH_AGCNT builds only)
  kSaSimt,     // self-attention unit: k_sa_qkv + k_sa_attn
  kSaTcQkv,    // self-attention unit: k_sa_affine + qkv conv on the single-tap k_tc_tcn + k_sa_attn
  kSaTcFused,  // self-attention unit: k_sa_affine + k_tc_sa (qkv conv and attention in one kernel: q, k, v never leave the SM)
};
// attention half of an adaptive graph conv, run before its mix: k_agcn_attn, k_attn_small or k_tc_attn
enum class AttnRoute : uint8_t { kNone, kSimt, kSmall, kTc };

struct Route {
  GcnRoute gcn = GcnRoute::kSimt;
  AttnRoute attn = AttnRoute::kNone;
  bool sa_out_tc = false;  // self-attention unit: output conv on the single-tap k_tc_tcn, else k_tcn_simt
  bool tcn_tc = false;     // temporal conv on k_tc_tcn / k_tc_tcn2 (tcn_on_pair), else k_tcn_simt
  bool block64 = false;    // a frame-by-frame walk runs graph conv + temporal conv as ONE kernel (k_tc_block64)
  bool gcn_tc() const {
    return gcn == GcnRoute::kTc || gcn == GcnRoute::kTcT || gcn == GcnRoute::kTcAgcn || gcn == GcnRoute::kTcAgcnt;
  }
};

struct BlockW {
  // host copies as loaded (BN already folded by the caller)
  std::vector<float> mix, gcn_w, gcn_b, tcn_w, res_w, tcn_b, att_w, att_b, sa_scale, sa_shift, sa_qkv_w, sa_qkv_b, sa_skip;
  Route route;
  // device, SIMT format (k-major fp32)
  float *d_gcn_w = nullptr, *d_gcn_b = nullptr, *d_tcn_w = nullptr, *d_res_w = nullptr, *d_tcn_b = nullptr;
  int *d_mix_ptr = nullptr, *d_mix_src = nullptr;
  float *d_mix_val = nullptr;
  float *d_att_w = nullptr, *d_att_b = nullptr, *d_adj = nullptr;  // adaptive graph conv: k-major embedding convs, dense A + graph_attn
  // self-attention unit: data_bn affine [cin][V], k-major qkv conv; its output conv lives in d_gcn_w / d_gcn_b
  float *d_sa_scale = nullptr, *d_sa_shift = nullptr, *d_sa_qkv_w = nullptr, *d_sa_qkv_b = nullptr, *d_res_w_sa = nullptr;
  __nv_bfloat16 *d_sa_w16 = nullptr;  // output conv (+ identity K-block) for the single-tap tcgen05 launch
  CUtensorMap map_sa_w, map_sa_w_half;
  __nv_bfloat16 *d_sa_fw16 = nullptr;  // qkv weights regrouped per head group: [items][hi: q, k, v | lo: same][cin]
  float *d_sa_fbias = nullptr;         // [items][96]
  CUtensorMap map_sa_fw;
  __nv_bfloat16 *d_sa_qw16 = nullptr;  // unfused qkv conv: [2*kSaQkvCols rows (hi, lo)][cin]
  float *d_sa_qbias = nullptr;
  CUtensorMap map_sa_q;
  int gcn_parts = 4;  // accumulator column groups of the tensor-core graph conv (3 or 4)
  bool gcn_folded = false;  // gcn_residual folded into W_0 on the host (every self link exactly 1): no residual rows, three groups
  // device, tensor-core format: [2*cout rows (hi, lo)][K] bf16
  __nv_bfloat16 *d_gcn_w16 = nullptr, *d_tcn_w16 = nullptr, *d_att_w16 = nullptr;
  CUtensorMap map_gcn_w, map_tcn_w, map_tcn_w_half, map_att_w;  // _half: box of cout/2 rows for the CTA-pair kernel
  CUtensorMap map_tcn_w_full;  // temporal-conv weights with a 2*cout-row box: hi and lo rows in one stacked slab
  // pre-mix graph conv weights of the fused block kernel: [2*cout rows (hi, lo)][gcnp_parts*cin], partition-major K
  int gcnp_parts = 3;
  __nv_bfloat16 *d_gcnp_w16 = nullptr;
  CUtensorMap map_gcnp_w;
  // channel-major graph conv (k_tc_gcnt, and k_tc_agcnt with always 4 parts): weights [2 planes][chunk of 128 channels][part][128]
  // x cin, tree coefficients
  int gcnt_parts = 4;
  __nv_bfloat16 *d_gcnt_w16 = nullptr;
  CUtensorMap map_gcnt_w;
  float gcnt_coef[3][32];
};

// The emission bookkeeping of a batch: frames entered, per block executions (n_in) and emissions (n_out), and vectors
// entered into the pooling window.  A function of the frame count alone (counters_at).
struct Counters {
  long long frame = 0, pool_n = 0;
  long long n_in[COSK_MAX_BLOCKS] = {}, n_out[COSK_MAX_BLOCKS] = {};
};

// A block's buffers in a batch (which of them are state and which scratch of the frame in flight: stream_state.cuh).
struct BlockBufs {
  ActBuf ring, out;  // temporal ring, block-output ring
  ActBuf sa;         // self-attention unit: attention rows of the frame in flight (1 slot), operand of the output conv
  // tensor-core qkv conv: normalised input rows; unfused (C = 64), the conv runs on the single-tap temporal-conv kernel
  // into q | k | v rows zero-padded to kSaQkvCols columns
  ActBuf sa_x, sa_q;
};

// The streams a handle steps: their geometry, ring sizes, buffers and counters.  alloc_batch builds one and free_batch
// frees it; whatever runs on state is handed the batch it runs on.  n_streams == 0: no batch (geometry and counters zero,
// ring sizes of time chunk 1, so the payload layout and the schedule can still be read from it).
struct Batch {
  long long n_streams = 0, n_tokens = 0, t_alloc = 0;
  int skel_per_tile = 0, tile_tokens = 0, n_tiles = 0;
  int dense_vp = 0;
  int tchunk = 1;  // time chunk: frames of one block processed per launch by cosk_steps (cosk_set_batch_ex)
  // slots of the temporal rings (8 + tchunk) and of the input / block-output rings (4 + tchunk)
  int R = kRingSlots, Ro = kOutSlots;
  ActBuf xin;
  BlockBufs blk[COSK_MAX_BLOCKS];
  float *d_pool_ring = nullptr;
  double *d_pool_sum = nullptr;
  float *d_qkv = nullptr;      // self-attention unit: q | k | v rows [t_alloc][2*dk + dv] of the frame in flight (fp32)
  float *d_dense = nullptr;    // adaptive graph conv: per-token mixing rows [t_alloc][3][dense_vp] of the frame in flight
  long long *d_idx = nullptr;  // [n_streams] stream indices of a per-stream state call (k_stream_state)
  int64_t state_bytes = 0;
  Counters cnt;
  int32_t last_flags[COSK_MAX_BLOCKS + 1] = {};  // cosk_last_schedule
};

struct ProfRec {
  int kind, block;
  cudaEvent_t ev;
};

}  // namespace

struct cosk_model {
  cosk_config cfg;
  int num_sms = 148;
  int gcn_transposed = 1;  // plain graph convs with cout in {128, 256}, cin in {64, 128} on a skeleton tree the kernel is compiled for run on
                           // k_tc_gcnt (channels on the TMEM lanes, adjacency contraction in registers); COSK_GCN_T=0: k_tc_gcn
  int agcn_transposed = 0;  // adaptive graph convs with cout in {128, 256}, cin in {64, 128}: dense mix on k_tc_agcnt.  OFF and not in the
                            // default build: the kernel was written after the round's GPU budget was spent and has never run on hardware
                            // (build with COSK_WITH_AGCNT=1, enable with COSK_AGCN_T=1, test with COSK_TEST_UNVERIFIED=1)
  int fuse_block = 1;  // 64 -> 64 identity-residual blocks: graph conv + temporal conv in one kernel per step (COSK_FUSE_BLOCK=0: two kernels)
  EncodeTiledFn encode = nullptr;
  std::vector<BlockW> blk;
  std::vector<float> h_bn_scale, h_bn_shift, h_fc_w, h_fc_b;
  float *d_bn_scale = nullptr, *d_bn_shift = nullptr, *d_fc_w = nullptr, *d_fc_b = nullptr;
  bool prepared = false;
  Batch batch;
  cudaEvent_t ev_idx = nullptr;    // recorded behind the last per-stream state call: the next one's index upload waits for it
  std::vector<long long> h_idx;    // host copy the index upload reads
  unsigned int *d_dbg = nullptr;
  unsigned int *h_dbg = nullptr;  // pinned copy of d_dbg, refreshed asynchronously after every call that emitted
  bool failed = false;            // a step stopped half way or the device watchdog fired: only cosk_reset / cosk_set_batch clear it
  unsigned long long *d_trace = nullptr;  // phase timers of the graph-conv kernel (COSK_TRACE=1)
  int64_t launches = 0;
  // profiling
  bool prof_on = false;
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  std::string err;
};

namespace {

// Every entry point runs on the handle's device and leaves the caller's current device as it found it
// (a host process may hold handles on several GPUs, and PyTorch tracks the current device per thread).
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

int fail(cosk_model *m, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (m) m->err = buf;
  return code;
}

#define CK(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e_ = (call);                                                                             \
    if (e_ != cudaSuccess)                                                                               \
      return fail(m, COSK_ERR_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
  } while (0)

template <typename T>
void dfree(T *&p) {
  if (p) cudaFree(p);
  p = nullptr;
}

// Frees what alloc_batch allocated, also when it stopped half way, and leaves `b` empty.
void free_batch(Batch &b) {
  dfree(b.xin.ptr);
  for (BlockBufs &k : b.blk)
    for (ActBuf *a : {&k.ring, &k.out, &k.sa, &k.sa_x, &k.sa_q}) dfree(a->ptr);
  dfree(b.d_qkv);
  dfree(b.d_pool_ring);
  dfree(b.d_pool_sum);
  dfree(b.d_dense);
  dfree(b.d_idx);
  b = Batch();
}

int make_map(cosk_model *m, CUtensorMap *map, void *base, uint64_t cols, uint64_t rows, uint32_t box_rows) {
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * sizeof(__nv_bfloat16)};
  cuuint32_t box[2] = {(cuuint32_t)kBK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = m->encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, gdim, gstride, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(m, COSK_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) cols=%llu rows=%llu", (int)r,
                                     (unsigned long long)cols, (unsigned long long)rows);
  return COSK_OK;
}

int alloc_act(cosk_model *m, Batch &bt, ActBuf &b, int slots, int c) {
  b.slots = slots;
  b.c = c;
  b.cs = round_up(c, 8);
  b.t_alloc = bt.t_alloc;
  CK(cudaMalloc(&b.ptr, b.bytes()));
  bt.state_bytes += (int64_t)b.bytes();
  b.has_map = false;
  if (b.cs % kBK == 0) {
    int rc = make_map(m, &b.map, b.ptr, (uint64_t)b.cs, (uint64_t)slots * 2 * b.t_alloc, kTileRows);
    if (rc) return rc;
    b.has_map = true;
  }
  return COSK_OK;
}

template <typename T>
int upload(cosk_model *m, T *&dst, const T *src, size_t n) {
  dfree(dst);
  CK(cudaMalloc(&dst, n * sizeof(T)));
  CK(cudaMemcpy(dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
  return COSK_OK;
}

// [rows][K] fp32 (K contiguous) -> k-major [K][rows]
std::vector<float> transpose(const float *w, int rows, int K) {
  std::vector<float> t((size_t)rows * K);
  for (int r = 0; r < rows; ++r)
    for (int k = 0; k < K; ++k) t[(size_t)k * rows + r] = w[(size_t)r * K + k];
  return t;
}

inline uint16_t f2bf(float x) {  // round-to-nearest-even, like __float2bfloat16_rn
  uint32_t u;
  memcpy(&u, &x, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
inline float bf2f(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

// [rows][K] fp32 -> [2*rows][K] bf16, per group of `group` rows (rows % group == 0): its hi rows, then its lo rows
std::vector<uint16_t> split_rows(const std::vector<float> &w, int rows, int K, int group) {
  std::vector<uint16_t> o((size_t)2 * rows * K);
  const size_t gk = (size_t)group * K;
  for (size_t i = 0; i < (size_t)rows * K; ++i) {
    const size_t hi = i + i / gk * gk;  // the rows of the groups before this one are stacked twice
    uint16_t h = f2bf(w[i]);
    o[hi] = h;
    o[hi + gk] = f2bf(w[i] - bf2f(h));
  }
  return o;
}

// split_rows of a [rows][K] weight matrix uploaded to `dst`, with a TMA map of `box`-row boxes
int upload_split(cosk_model *m, __nv_bfloat16 *&dst, CUtensorMap *map, const std::vector<float> &w, int rows, int K, uint32_t box,
                 int group = 0) {
  const std::vector<uint16_t> s = split_rows(w, rows, K, group ? group : rows);
  int rc = upload(m, reinterpret_cast<uint16_t *&>(dst), s.data(), s.size());
  return rc ? rc : make_map(m, map, dst, (uint64_t)K, (uint64_t)2 * rows, box);
}

// Graph-conv weights [cout][(3 + res_conv) * cin] regrouped per part for the tensor-core kernels: row
// (o / group) * (P * group) + part * group + o % group holds W_part of output channel o, K = cin.  Part 3, when P = 4, is the
// gcn_residual branch: the folded 1x1 conv when cin != cout, else the identity matrix.  `fold`: the residual is added into W_0
// instead (every self link exactly 1).
std::vector<float> regroup_parts(const std::vector<float> &gcn_w, int cin, int cout, int group, int P, bool fold) {
  const bool res_conv = cin != cout;
  const size_t Kg = (size_t)(3 + res_conv) * cin;
  std::vector<float> re((size_t)P * cout * cin, 0.f);
  for (int o = 0; o < cout; ++o)
    for (int part = 0; part < P; ++part) {
      float *row = &re[((size_t)(o / group) * (P * group) + (size_t)part * group + (o % group)) * cin];
      if (part < 3 || res_conv) memcpy(row, &gcn_w[(size_t)o * Kg + (size_t)part * cin], sizeof(float) * cin);
      else row[o] = 1.0f;
      if (fold && part == 0) {
        if (res_conv)
          for (int k = 0; k < cin; ++k) row[k] += gcn_w[(size_t)o * Kg + (size_t)3 * cin + k];
        else
          row[o] += 1.0f;
      }
    }
  return re;
}

// Does the mixing matrix have exactly the sparsity of the skeleton tree k_tc_gcnt is compiled for (partition 1 = one entry
// per vertex, from its parent; partition 2 = entries from a vertex's children)?  Fills the kernel's coefficients.
bool tree_coefs(const std::vector<float> &mix, int V, float coef[3][32]) {
  auto parent = [&](int w) { return V == 25 ? skel_parent<25>(w) : skel_parent<18>(w); };
  bool tree = true;
  memset(coef, 0, sizeof(float) * 3 * 32);
  for (int v = 0; v < V; ++v)
    for (int w = 0; w < V; ++w) {
      const float a0 = mix[((size_t)0 * V + v) * V + w], a1 = mix[((size_t)1 * V + v) * V + w], a2 = mix[((size_t)2 * V + v) * V + w];
      if (v == w) coef[0][w] = a0;
      if (a1 != 0.f) {
        if (parent(w) == v) coef[1][w] = a1;
        else tree = false;
      }
      if (a2 != 0.f) {
        if (parent(v) == w) coef[2][v] = a2;
        else tree = false;
      }
    }
  return tree;
}

bool tc_width(int c) { return c == 64 || c == 128 || c == 256; }

// Narrow first layer (cin <= 8): k_gcn_small keeps the weights and the mixed inputs of a tile in shared memory, and the
// adaptive one computes its embeddings per thread (k_attn_small).
bool gcn_small(const cosk_model *m, const cosk_block_cfg &bc) {
  const int res_conv = bc.cin != bc.cout ? 1 : 0;
  return m->cfg.path == COSK_PATH_AUTO && bc.cin <= 8 && res_conv && bc.cout % 32 == 0 && (3 + res_conv) * bc.cin <= kSmallKMax;
}
bool attn_small(const cosk_model *m, const cosk_block_cfg &bc) {
  return bc.gconv == COSK_GCONV_ADAPTIVE && m->cfg.path == COSK_PATH_AUTO && bc.cin <= 8 && bc.cout == 64 &&
         (m->cfg.vertices == 25 || m->cfg.vertices == 18);
}

// The tensor-core temporal conv takes the residual as extra K-blocks of its GEMM (folded strided conv, or identity weights
// for the narrow layers) instead of epilogue loads.
bool tcn_res_kblock(const cosk_block_cfg &bc) {
  return bc.res_kind == COSK_RES_CONV || (bc.res_kind == COSK_RES_IDENTITY && bc.cout <= 128);
}

int prepare(cosk_model *m) {
  const cosk_config &c = m->cfg;
  const int V = c.vertices;
  if (c.data_bn) {
    size_t n = (size_t)c.persons * V * c.c_in;
    if (m->h_bn_scale.size() != n || m->h_bn_shift.size() != n) return fail(m, COSK_ERR_STATE, "data_bn weights missing");
    int rc = upload(m, m->d_bn_scale, m->h_bn_scale.data(), n);
    if (rc) return rc;
    rc = upload(m, m->d_bn_shift, m->h_bn_shift.data(), n);
    if (rc) return rc;
  }
  if (c.classes > 0) {
    size_t n = (size_t)c.classes * c.blocks[c.n_blocks - 1].cout;
    if (m->h_fc_w.size() != n || m->h_fc_b.size() != (size_t)c.classes) return fail(m, COSK_ERR_STATE, "fc weights missing");
    int rc = upload(m, m->d_fc_w, m->h_fc_w.data(), n);
    if (rc) return rc;
    rc = upload(m, m->d_fc_b, m->h_fc_b.data(), (size_t)c.classes);
    if (rc) return rc;
  }
  for (int i = 0; i < c.n_blocks; ++i) {
    const cosk_block_cfg &bc = c.blocks[i];
    BlockW &b = m->blk[i];
    const int res_conv = bc.cin != bc.cout ? 1 : 0;
    const bool attention = bc.gconv == COSK_GCONV_ATTENTION;
    const int Kg = attention ? bc.cout : (3 + res_conv) * bc.cin, Kt = kTaps * bc.cout;
    if (attention) {
      const int nq = 2 * (bc.cout / 4) + bc.cout;
      if (b.sa_scale.size() != (size_t)bc.cin * V || b.sa_shift.size() != (size_t)bc.cin * V)
        return fail(m, COSK_ERR_STATE, "block%d.sa.in_scale / in_shift missing or wrong size", i);
      if (b.sa_qkv_w.size() != (size_t)nq * bc.cin || b.sa_qkv_b.size() != (size_t)nq)
        return fail(m, COSK_ERR_STATE, "block%d.sa.qkv.w / qkv.b missing or wrong size", i);
      if (!res_conv && b.sa_skip.size() != (size_t)bc.cout) return fail(m, COSK_ERR_STATE, "block%d.sa.skip_scale missing", i);
      b.mix.assign((size_t)3 * V * V, 0.f);  // the unit does not mix with the adjacency (only_attention)
    }
    if (b.mix.size() != (size_t)3 * V * V) return fail(m, COSK_ERR_STATE, "block%d.mix missing", i);
    if (b.gcn_w.size() != (size_t)bc.cout * Kg) return fail(m, COSK_ERR_STATE, "block%d.gcn.w missing or wrong size", i);
    if (b.gcn_b.size() != (size_t)bc.cout) return fail(m, COSK_ERR_STATE, "block%d.gcn.b missing", i);
    if (b.tcn_w.size() != (size_t)bc.cout * Kt) return fail(m, COSK_ERR_STATE, "block%d.tcn.w missing", i);
    if (b.tcn_b.size() != (size_t)bc.cout) return fail(m, COSK_ERR_STATE, "block%d.tcn.b missing", i);
    if (bc.res_kind == COSK_RES_CONV && b.res_w.size() != (size_t)bc.cout * bc.cin)
      return fail(m, COSK_ERR_STATE, "block%d.res.w missing", i);
    const bool adaptive = bc.gconv == COSK_GCONV_ADAPTIVE;
    if (adaptive) {
      const int ic = bc.cout / 4;  // coff_embedding = 4, models/a_gcn/a_gcn.py:13-14
      if (b.att_w.size() != (size_t)6 * ic * bc.cin || b.att_b.size() != (size_t)6 * ic)
        return fail(m, COSK_ERR_STATE, "block%d.att.w / att.b missing or wrong size", i);
    }
    // CSR of A * graph_attn over (partition, output vertex)
    std::vector<int> ptr(3 * V + 1, 0), src;
    std::vector<float> val;
    bool mix_diag0 = true;  // partition 0 has only self links
    for (int p = 0; p < 3; ++p)
      for (int w = 0; w < V; ++w) {
        for (int v = 0; v < V; ++v) {
          float a = b.mix[((size_t)p * V + v) * V + w];
          if (a != 0.f) {
            src.push_back(v);
            val.push_back(a);
            if (p == 0 && v != w) mix_diag0 = false;
          }
        }
        ptr[p * V + w + 1] = (int)src.size();
      }
    // most non-zeros of partitions 1 and 2 together, and of one of them, for one output vertex
    int mix_max_row12 = 0, part_max = 0;
    for (int w = 0; w < V; ++w) {
      const int n1 = ptr[V + w + 1] - ptr[V + w], n2 = ptr[2 * V + w + 1] - ptr[2 * V + w];
      mix_max_row12 = std::max(mix_max_row12, n1 + n2);
      part_max = std::max({part_max, n1, n2});
    }
    // Every self link exactly 1 (A_0 = I with graph_attn's diagonal at 1, the reference initialisation): the own-row term of
    // partition 0 and the gcn_residual branch act on the same rows, x W_0^T + x R^T = x (W_0 + R)^T, so the plain tensor-core
    // graph convs add the residual (identity or folded conv) into W_0 on the host and drop a part: a quarter fewer MMAs and
    // TMEM reads, no residual rows fetched.  Trained self-link coefficients keep the four-part form.
    bool unit_diag = !adaptive && mix_diag0;
    for (int w0 = 0; unit_diag && w0 < V; ++w0) unit_diag = (ptr[w0 + 1] - ptr[w0] == 1 && val[ptr[w0]] == 1.0f);
    if (src.empty()) {
      src.push_back(0);
      val.push_back(0.f);
    }
    int rc;
    if ((rc = upload(m, b.d_mix_ptr, ptr.data(), ptr.size()))) return rc;
    if ((rc = upload(m, b.d_mix_src, src.data(), src.size()))) return rc;
    if ((rc = upload(m, b.d_mix_val, val.data(), val.size()))) return rc;
    // SIMT weights
    std::vector<float> t = transpose(b.gcn_w.data(), bc.cout, Kg);
    if ((rc = upload(m, b.d_gcn_w, t.data(), t.size()))) return rc;
    if ((rc = upload(m, b.d_gcn_b, b.gcn_b.data(), b.gcn_b.size()))) return rc;
    t = transpose(b.tcn_w.data(), bc.cout, Kt);
    if ((rc = upload(m, b.d_tcn_w, t.data(), t.size()))) return rc;
    if ((rc = upload(m, b.d_tcn_b, b.tcn_b.data(), b.tcn_b.size()))) return rc;
    if (bc.res_kind == COSK_RES_CONV) {
      t = transpose(b.res_w.data(), bc.cout, bc.cin);
      if ((rc = upload(m, b.d_res_w, t.data(), t.size()))) return rc;
    }
    if (adaptive) {
      t = transpose(b.att_w.data(), 6 * (bc.cout / 4), bc.cin);
      if ((rc = upload(m, b.d_att_w, t.data(), t.size()))) return rc;
      if ((rc = upload(m, b.d_att_b, b.att_b.data(), b.att_b.size()))) return rc;
      if ((rc = upload(m, b.d_adj, b.mix.data(), b.mix.size()))) return rc;
    }

    // The route: which kernels serve this block.
    Route &rt = b.route;
    rt = Route();
    const bool want_tc = c.path == COSK_PATH_AUTO;
    const bool skel_v = V == 25 || V == 18;  // the skeletons the dense-mix and channel-major kernels are instantiated for
    const bool t_shape = (bc.cout == 128 || bc.cout == 256) && (bc.cin == 64 || bc.cin == 128) && skel_v;  // channel-major kernels
    bool tc_gcn = false;  // graph conv (adaptive: its mix) on the tensor cores, with weights in the k_tc_gcn layout
    if (adaptive)
      tc_gcn = want_tc && bc.cout % 64 == 0 && bc.cout <= 256 && bc.cin % kBK == 0 && skel_v;
    else if (!attention)
      tc_gcn = want_tc && bc.cout % 64 == 0 && bc.cout <= 256 && bc.cin % kBK == 0 && mix_max_row12 <= kMixSlots && mix_diag0;
    if (attention) {
      // The fused kernel has eight epilogue warps per SM for the attention math: a win where the q | k | v round trip
      // dominates (C >= 128), a loss for the 64-channel unit, whose eight tiny heads want the separate kernel's occupancy.
      const bool tc_qkv = want_tc && bc.cin % kBK == 0 && tc_width(bc.cout);
      rt.gcn = !tc_qkv ? GcnRoute::kSaSimt : bc.cout >= 128 ? GcnRoute::kSaTcFused : GcnRoute::kSaTcQkv;
      rt.sa_out_tc = want_tc && tc_width(bc.cout);
    } else if (adaptive) {
      rt.attn = tc_gcn && tc_width(bc.cout) ? AttnRoute::kTc : attn_small(m, bc) ? AttnRoute::kSmall : AttnRoute::kSimt;
      if (tc_gcn) rt.gcn = kAgcntBuilt && m->agcn_transposed && t_shape ? GcnRoute::kTcAgcnt : GcnRoute::kTcAgcn;
      else rt.gcn = gcn_small(m, bc) ? GcnRoute::kSmall : GcnRoute::kSimt;
    } else if (tc_gcn) {
      rt.gcn = m->gcn_transposed && t_shape && tree_coefs(b.mix, V, b.gcnt_coef) ? GcnRoute::kTcT : GcnRoute::kTc;
    } else {
      rt.gcn = gcn_small(m, bc) ? GcnRoute::kSmall : GcnRoute::kSimt;
    }
    rt.tcn_tc = want_tc && tc_width(bc.cout) && (bc.res_kind != COSK_RES_CONV || bc.cin % kBK == 0);
    // one kernel per block step: 64 -> 64 blocks with the identity residual riding in both GEMMs; the sources per
    // (partition >= 1, output vertex) must fit the register CSR of its pre-mix graph conv
    rt.block64 = m->fuse_block && tc_gcn && bc.gconv == COSK_GCONV_PLAIN && part_max <= kPartSrcMax && bc.cin == 64 &&
                bc.cout == 64 && bc.stride == 1 && bc.res_kind == COSK_RES_IDENTITY && rt.tcn_tc && tcn_res_kblock(bc);

    // Tensor-core weights of the route.
    if (tc_gcn) {
      // k_tc_gcn: 64-row groups.  The identity gcn_residual rides in the GEMM (fourth part) except for the 256-channel layers,
      // where the mix warps have the slack to add the input rows and the narrower accumulator saves MMA columns and TMEM
      // reads (measured -8 %).  (adaptive: 4 parts need the single-stage layout, so the identity rides along only when one
      // K-block is all there is)
      const bool ident_mma = bc.cin < 256;
      b.gcn_folded = unit_diag;
      const int P = b.gcn_parts = adaptive ? ((res_conv || bc.cin == kBK) ? 4 : 3) : (unit_diag ? 3 : ((res_conv || ident_mma) ? 4 : 3));
      if ((rc = upload_split(m, b.d_gcn_w16, &b.map_gcn_w, regroup_parts(b.gcn_w, bc.cin, bc.cout, 64, P, unit_diag), P * bc.cout,
                             bc.cin, (uint32_t)(P * 64))))
        return rc;
    }
    if (rt.gcn == GcnRoute::kTcT || rt.gcn == GcnRoute::kTcAgcnt) {
      // channel-major layout, 128-row groups, the residual folded as for k_tc_gcn (k_tc_agcnt: never, always four parts)
      const int P = b.gcnt_parts = b.gcn_folded ? 3 : 4;
      if ((rc = upload_split(m, b.d_gcnt_w16, &b.map_gcnt_w, regroup_parts(b.gcn_w, bc.cin, bc.cout, 128, P, b.gcn_folded),
                             P * bc.cout, bc.cin, 128u)))
        return rc;
    }
    if (rt.block64) {
      // Pre-mix form.  K-blocks in the order the mix warps fill their A slots: the plain input rows (gcn_residual weights:
      // folded 1x1 conv or identity; plus W_0 when every self link is exactly 1, so that x and 1*x share one part),
      // [W_0 on a0*x], W_1, W_2
      const int P = b.gcnp_parts = unit_diag ? 3 : 4;
      const int K = P * bc.cin;
      std::vector<float> w((size_t)bc.cout * K, 0.f);
      for (int o = 0; o < bc.cout; ++o) {
        float *row = &w[(size_t)o * K];
        const float *src = &b.gcn_w[(size_t)o * Kg];
        if (res_conv) memcpy(row, src + 3 * bc.cin, sizeof(float) * bc.cin);
        else row[o] = 1.0f;
        if (unit_diag) {
          for (int k = 0; k < bc.cin; ++k) row[k] += src[k];
          memcpy(row + bc.cin, src + bc.cin, sizeof(float) * 2 * bc.cin);
        } else {
          memcpy(row + bc.cin, src, sizeof(float) * 3 * bc.cin);
        }
      }
      if ((rc = upload_split(m, b.d_gcnp_w16, &b.map_gcnp_w, w, bc.cout, K, (uint32_t)std::min(2 * bc.cout, 256)))) return rc;
    }
    if (attention) {
      std::vector<float> tq = transpose(b.sa_qkv_w.data(), 2 * (bc.cout / 4) + bc.cout, bc.cin);
      if ((rc = upload(m, b.d_sa_qkv_w, tq.data(), tq.size()))) return rc;
      if ((rc = upload(m, b.d_sa_qkv_b, b.sa_qkv_b.data(), b.sa_qkv_b.size()))) return rc;
      if ((rc = upload(m, b.d_sa_scale, b.sa_scale.data(), b.sa_scale.size()))) return rc;
      if ((rc = upload(m, b.d_sa_shift, b.sa_shift.data(), b.sa_shift.size()))) return rc;
      if (rt.gcn == GcnRoute::kSaTcQkv) {
        const int nq = 2 * (bc.cout / 4) + bc.cout;
        std::vector<float> w((size_t)kSaQkvCols * bc.cin, 0.f), bb((size_t)kSaQkvCols, 0.f);  // rows nq.. stay zero
        memcpy(w.data(), b.sa_qkv_w.data(), sizeof(float) * nq * bc.cin);
        memcpy(bb.data(), b.sa_qkv_b.data(), sizeof(float) * nq);
        if ((rc = upload_split(m, b.d_sa_qw16, &b.map_sa_q, w, kSaQkvCols, bc.cin, (uint32_t)kSaQkvCols))) return rc;
        if ((rc = upload(m, b.d_sa_qbias, bb.data(), bb.size()))) return rc;
      }
      if (rt.gcn == GcnRoute::kSaTcFused) {
        const int dk = bc.cout / 4, dvh = bc.cout / 8, dkh = dk / 8, G = 64 / dvh, items = 8 / G;
        std::vector<float> w((size_t)items * 96 * bc.cin), bb((size_t)items * 96);
        for (int it = 0; it < items; ++it)
          for (int r = 0; r < 96; ++r) {
            int src;  // row of the [q | k | v] conv this column of the item comes from
            if (r < 16) src = (it * G + r / dkh) * dkh + r % dkh;                       // q of head it*G + r/dkh
            else if (r < 32) src = dk + (it * G + (r - 16) / dkh) * dkh + (r - 16) % dkh;  // k
            else src = 2 * dk + (it * G + (r - 32) / dvh) * dvh + (r - 32) % dvh;          // v
            memcpy(&w[((size_t)it * 96 + r) * bc.cin], &b.sa_qkv_w[(size_t)src * bc.cin], sizeof(float) * bc.cin);
            bb[(size_t)it * 96 + r] = b.sa_qkv_b[src];
          }
        if ((rc = upload_split(m, b.d_sa_fw16, &b.map_sa_fw, w, items * 96, bc.cin, 192u, 96))) return rc;  // hi | lo per item
        if ((rc = upload(m, b.d_sa_fbias, bb.data(), bb.size()))) return rc;
      }
      // The skip connection is added before the unit's bn, so it enters scaled per channel: a diagonal "residual conv".
      if (!res_conv) {
        std::vector<float> diag((size_t)bc.cin * bc.cout, 0.f);  // k-major [cin][cout]
        for (int r = 0; r < bc.cout; ++r) diag[(size_t)r * bc.cout + r] = b.sa_skip[r];
        if ((rc = upload(m, b.d_res_w_sa, diag.data(), diag.size()))) return rc;
      }
      // output conv on the temporal-conv kernel with a single tap: [W0 | diag(skip scale) K-block on the input rows]
      if (rt.sa_out_tc) {
        const int Kr = res_conv ? 0 : bc.cin, K0 = bc.cout;
        std::vector<float> cat((size_t)bc.cout * (K0 + Kr), 0.f);
        for (int r = 0; r < bc.cout; ++r) {
          memcpy(&cat[(size_t)r * (K0 + Kr)], &b.gcn_w[(size_t)r * K0], sizeof(float) * K0);
          if (Kr) cat[(size_t)r * (K0 + Kr) + K0 + r] = b.sa_skip[r];
        }
        if ((rc = upload_split(m, b.d_sa_w16, &b.map_sa_w, cat, bc.cout, K0 + Kr, (uint32_t)bc.cout))) return rc;
        if ((rc = make_map(m, &b.map_sa_w_half, b.d_sa_w16, (uint64_t)(K0 + Kr), (uint64_t)2 * bc.cout, (uint32_t)bc.cout / 2))) return rc;
      }
    }
    if (rt.attn == AttnRoute::kTc) {
      // per partition: hi rows of (theta, phi), then their lo rows -- one stacked operand of 4*IC rows
      const int ic = bc.cout / 4;
      if ((rc = upload_split(m, b.d_att_w16, &b.map_att_w, b.att_w, 6 * ic, bc.cin, (uint32_t)(4 * ic), 2 * ic))) return rc;
    }
    if (rt.tcn_tc) {
      // The delayed residual x_{n-4} is streamed through the operand ring like a tenth tap: with the folded
      // strided 1x1 conv as its weights (layers 5 and 8), or -- for the identity residual of the HBM-bound
      // narrow layers -- with identity weights (exact under the split products), which removes every
      // latency-bound load from the epilogue.  The 256-channel layers are tensor-bound and keep the add.
      const int Kr = tcn_res_kblock(bc) ? bc.cin : 0;
      std::vector<float> cat((size_t)bc.cout * (Kt + Kr));
      for (int r = 0; r < bc.cout; ++r) {
        memcpy(&cat[(size_t)r * (Kt + Kr)], &b.tcn_w[(size_t)r * Kt], sizeof(float) * Kt);
        if (bc.res_kind == COSK_RES_CONV) memcpy(&cat[(size_t)r * (Kt + Kr) + Kt], &b.res_w[(size_t)r * Kr], sizeof(float) * Kr);
        else
          for (int k = 0; k < Kr; ++k) cat[(size_t)r * (Kt + Kr) + Kt + k] = k == r ? 1.0f : 0.0f;
      }
      if ((rc = upload_split(m, b.d_tcn_w16, &b.map_tcn_w, cat, bc.cout, Kt + Kr, (uint32_t)bc.cout))) return rc;
      if ((rc = make_map(m, &b.map_tcn_w_half, b.d_tcn_w16, (uint64_t)(Kt + Kr), (uint64_t)2 * bc.cout, (uint32_t)bc.cout / 2)))
        return rc;
      if (bc.cout <= 128 &&
          (rc = make_map(m, &b.map_tcn_w_full, b.d_tcn_w16, (uint64_t)(Kt + Kr), (uint64_t)2 * bc.cout, (uint32_t)(2 * bc.cout))))
        return rc;
    }
  }
  m->prepared = true;
  return COSK_OK;
}

// Zeroes every state buffer (not the counters).
int zero_buffers(cosk_model *m, const Batch &bt, cudaStream_t s) {
  CK(cudaMemsetAsync(bt.xin.ptr, 0, bt.xin.bytes(), s));
  for (int i = 0; i < m->cfg.n_blocks; ++i) {
    CK(cudaMemsetAsync(bt.blk[i].ring.ptr, 0, bt.blk[i].ring.bytes(), s));
    CK(cudaMemsetAsync(bt.blk[i].out.ptr, 0, bt.blk[i].out.bytes(), s));
  }
  if (m->cfg.classes > 0) {
    const size_t cl = (size_t)m->cfg.blocks[m->cfg.n_blocks - 1].cout;
    CK(cudaMemsetAsync(bt.d_pool_ring, 0, (size_t)m->cfg.pool_size * bt.n_streams * cl * sizeof(float), s));
    CK(cudaMemsetAsync(bt.d_pool_sum, 0, (size_t)bt.n_streams * cl * sizeof(double), s));
  }
  return COSK_OK;
}

// Zeroes the batch's buffers and counters, and clears the handle's watchdog word and failure latch.
int zero_state(cosk_model *m, Batch &bt, cudaStream_t s) {
  int rc = zero_buffers(m, bt, s);
  if (rc) return rc;
  CK(cudaMemsetAsync(m->d_dbg, 0, 4 * sizeof(unsigned int), s));
  if (m->h_dbg) m->h_dbg[0] = 0;
  m->failed = false;
  bt.cnt = Counters();
  std::fill(std::begin(bt.last_flags), std::end(bt.last_flags), 0);
  return COSK_OK;
}

// Every kernel goes through here: the launch carries the programmatic-stream-serialization attribute (PDL; the kernels
// call griddepcontrol.wait before touching their predecessor's output): +16 % at 256 streams, +4 % at 1024, neutral at 4096.
template <typename... KArgs, typename... Args>
cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args &&...args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

int prof_mark(cosk_model *m, int kind, int block, cudaStream_t s) {
  if (!m->prof_on) return COSK_OK;
  if (m->ev_used == m->ev_pool.size()) {
    cudaEvent_t e;
    CK(cudaEventCreate(&e));
    m->ev_pool.push_back(e);
  }
  cudaEvent_t e = m->ev_pool[m->ev_used++];
  CK(cudaEventRecord(e, s));
  m->prof.push_back({kind, block, e});
  return COSK_OK;
}

// Persistent kernels: one CTA per work item, at most one per SM.
int persistent_grid(const cosk_model *m, int items) { return std::min(items, m->num_sms); }

// The launchers size their grids for the (frame, tile) work items of `args`: n_tiles * n_frames.
template <int COUT>
int launch_tc_tcn(cosk_model *m, const Batch &bt, const TcTcnArgs &args, cudaStream_t s) {
  const dim3 grid(persistent_grid(m, bt.n_tiles * args.n_frames));
  CK(launch_k(k_tc_tcn<COUT>, grid, dim3(256), TcTcnCfg<COUT>::kSmemBytes, s, args));
  return COSK_OK;
}
template <int COUT>
int launch_tc_tcn2(cosk_model *m, const Batch &bt, const TcTcnArgs &args, cudaStream_t s) {
  // CTA pairs: one cluster of 2 per pair of adjacent token tiles, at most one CTA per SM
  const int n_pairs = (bt.n_tiles + 1) / 2 * args.n_frames;
  const int max_clusters = m->num_sms / 2;
  const int grid = 2 * (n_pairs < max_clusters ? n_pairs : max_clusters);
  CK(launch_k(k_tc_tcn2<COUT>, dim3(grid), dim3(256), TcTcn2Cfg<COUT>::kSmemBytes, s, args));
  return COSK_OK;
}
template <int P, int STAGES>
int launch_tc_gcn(cosk_model *m, const Batch &bt, const TcGcnArgs &args, cudaStream_t s) {
  const dim3 grid(persistent_grid(m, bt.n_tiles * args.n_frames));
  if (m->d_trace) CK(launch_k(k_tc_gcn<P, STAGES, true>, grid, dim3(512), TcGcnCfg<P, STAGES>::kSmemBytes, s, args));
  else CK(launch_k(k_tc_gcn<P, STAGES, false>, grid, dim3(512), TcGcnCfg<P, STAGES>::kSmemBytes, s, args));
  return COSK_OK;
}

template <int P, int STAGES, int V>
int launch_tc_agcn(cosk_model *m, const Batch &bt, const TcGcnArgs &args, cudaStream_t s) {
  CK(launch_k(k_tc_agcn<P, STAGES, V>, dim3(persistent_grid(m, bt.n_tiles)), dim3(512), TcAgcnCfg<P, STAGES>::kSmemBytes, s, args));
  return COSK_OK;
}

template <int IC, int V>
int launch_tc_attn(cosk_model *m, const Batch &bt, const TcAttnArgs &args, cudaStream_t s) {
  CK(launch_k(k_tc_attn<IC, V>, dim3(persistent_grid(m, bt.n_tiles)), dim3(384), TcAttnCfg<IC, V>::kSmemBytes, s, args));
  return COSK_OK;
}

int set_smem_attrs(cosk_model *m) {
  CK(cudaFuncSetAttribute(k_agcn_attn, cudaFuncAttributeMaxDynamicSharedMemorySize, kAttnMaxSmem));
  CK(cudaFuncSetAttribute(k_tc_sa<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSaCfg<16>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_sa<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSaCfg<32>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_attn<16, 25>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAttnCfg<16, 25>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_attn<32, 25>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAttnCfg<32, 25>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_attn<64, 25>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAttnCfg<64, 25>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_attn<16, 18>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAttnCfg<16, 18>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_attn<32, 18>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAttnCfg<32, 18>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_attn<64, 18>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAttnCfg<64, 18>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_agcn<4, 1, 25>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAgcnCfg<4, 1>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_agcn<3, 2, 25>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAgcnCfg<3, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_agcn<4, 1, 18>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAgcnCfg<4, 1>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_agcn<3, 2, 18>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAgcnCfg<3, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_tcn<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcTcnCfg<64>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_tcn<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcTcnCfg<128>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_tcn<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcTcnCfg<256>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_tcn2<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcTcn2Cfg<128>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_tcn2<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcTcn2Cfg<256>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcn<3, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcnCfg<3, 1>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcn<3, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcnCfg<3, 1>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcn<3, 2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcnCfg<3, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcn<3, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcnCfg<3, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcn<4, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcnCfg<4, 1>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcn<4, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcnCfg<4, 1>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcn<4, 2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcnCfg<4, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcn<4, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcnCfg<4, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_block64, cudaFuncAttributeMaxDynamicSharedMemorySize, TcBlockCfg::kSmemBytes));
#ifdef COSK_WITH_AGCNT
  CK(cudaFuncSetAttribute(k_tc_agcnt<25, 1, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAgcntCfg<25, 1>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_agcnt<25, 2, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAgcntCfg<25, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_agcnt<25, 2, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAgcntCfg<25, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_agcnt<18, 1, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAgcntCfg<18, 1>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_agcnt<18, 2, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAgcntCfg<18, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_agcnt<18, 2, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcAgcntCfg<18, 2>::kSmemBytes));
#endif
  CK(cudaFuncSetAttribute(k_tc_gcnt<25, 1, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcntCfg<25, 1>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcnt<25, 2, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcntCfg<25, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcnt<25, 2, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcntCfg<25, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcnt<18, 1, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcntCfg<18, 1>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcnt<18, 2, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcntCfg<18, 2>::kSmemBytes));
  CK(cudaFuncSetAttribute(k_tc_gcnt<18, 2, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcGcntCfg<18, 2>::kSmemBytes));
  return COSK_OK;
}

// Ring slots of a launch over consecutive executions: frame f of the launch is frame n + f * step of the stream.
RingWalk ring_walk(long long n, int step, int slots) {
  RingWalk w;
  w.slot0 = mod_slot(n, slots), w.step = step, w.slots = slots;
  return w;
}

// Arguments of the tensor-core graph convs for n_frames executions of block i: frame f reads slot in_walk.slot(f) of `in` and
// writes slot ring_walk.slot(f) of the block's temporal ring.
TcGcnArgs make_gcn_args(cosk_model *m, const Batch &bt, int i, const ActBuf &in, int n_frames, RingWalk in_walk, RingWalk ring_walk) {
  const cosk_block_cfg &bc = m->cfg.blocks[i];
  BlockW &b = m->blk[i];
  const ActBuf &ring = bt.blk[i].ring;
  const bool batched = n_frames > 1;  // pointers at slot 0 of their rings, the slots from the walks
  const int in_slot = batched ? 0 : in_walk.slot0, ring_slot = batched ? 0 : ring_walk.slot0;
  TcGcnArgs a;
  a.tm_x = in.map;
  a.tm_w = b.map_gcn_w;
  a.x_row = (int)in.row_hi(in_slot);
  a.t_alloc = (int)bt.t_alloc;
  a.cin = bc.cin;
  a.cout = bc.cout;
  a.V = m->cfg.vertices;
  a.n_tiles = bt.n_tiles;
  a.tile_tokens = bt.tile_tokens;
  a.n_tokens = bt.n_tokens;
  a.mix_ptr = b.d_mix_ptr;
  a.mix_src = b.d_mix_src;
  a.mix_val = b.d_mix_val;
  a.trace = m->d_trace;
  a.epi.bias = b.d_gcn_b;
  const bool epi_res = b.gcn_parts == 3 && !b.gcn_folded;  // identity gcn_residual added from the input rows by the epilogue
  a.epi.r_hi = epi_res ? in.hi(in_slot) : nullptr;
  a.epi.r_lo = epi_res ? in.lo(in_slot) : nullptr;
  a.epi.cs_r = in.cs;
  a.epi.y_hi = ring.hi(ring_slot);
  a.epi.y_lo = ring.lo(ring_slot);
  a.epi.cs_out = ring.cs;
  a.dbg = m->d_dbg;
  a.dense = bt.d_dense;
  a.dense_ld = 3 * bt.dense_vp;
  a.dense_vp = bt.dense_vp;
  if (batched) {
    a.n_frames = n_frames;
    a.slot_rows = (int)(2 * bt.t_alloc);
    a.in_walk = in_walk;
    a.out_walk = ring_walk;
    a.in_slot_elems = in.slot_elems();
    a.out_slot_elems = ring.slot_elems();
  }
  return a;
}

// k_tc_gcnt: `a` as for k_tc_gcn (per-frame or time-batched); work items are pairs of adjacent tiles
int launch_tc_gcnt(cosk_model *m, const Batch &bt, int i, TcGcnArgs a, cudaStream_t s) {
  const cosk_block_cfg &bc = m->cfg.blocks[i];
  const BlockW &b = m->blk[i];
  TcGcntArgs t;
  t.g = a;
  t.g.tm_w = b.map_gcnt_w;
  t.g.epi.r_hi = t.g.epi.r_lo = nullptr;  // gcn_residual always rides in the GEMM here
  memcpy(t.coef, b.gcnt_coef, sizeof t.coef);
  t.n_parts = b.gcnt_parts;
  const dim3 grid(persistent_grid(m, ((bt.n_tiles + 1) / 2) * a.n_frames)), block(384);
  const bool v25 = m->cfg.vertices == 25;
  if (bc.cout == 128 && bc.cin == 64) {
    if (v25) CK(launch_k(k_tc_gcnt<25, 1, 128>, grid, block, TcGcntCfg<25, 1>::kSmemBytes, s, t));
    else CK(launch_k(k_tc_gcnt<18, 1, 128>, grid, block, TcGcntCfg<18, 1>::kSmemBytes, s, t));
  } else if (bc.cout == 128) {
    if (v25) CK(launch_k(k_tc_gcnt<25, 2, 128>, grid, block, TcGcntCfg<25, 2>::kSmemBytes, s, t));
    else CK(launch_k(k_tc_gcnt<18, 2, 128>, grid, block, TcGcntCfg<18, 2>::kSmemBytes, s, t));
  } else {
    if (v25) CK(launch_k(k_tc_gcnt<25, 2, 256>, grid, block, TcGcntCfg<25, 2>::kSmemBytes, s, t));
    else CK(launch_k(k_tc_gcnt<18, 2, 256>, grid, block, TcGcntCfg<18, 2>::kSmemBytes, s, t));
  }
  return COSK_OK;
}

// k_tc_agcnt: dense mix of the adaptive graph conv, work items are single tiles
int launch_tc_agcnt(cosk_model *m, const Batch &bt, int i, TcGcnArgs a, cudaStream_t s) {
#ifndef COSK_WITH_AGCNT
  (void)bt, (void)i, (void)a, (void)s;
  return fail(m, COSK_ERR_STATE, "k_tc_agcnt is not compiled in (build with -DCOSK_WITH_AGCNT)");
#else
  const cosk_block_cfg &bc = m->cfg.blocks[i];
  const BlockW &b = m->blk[i];
  TcGcntArgs t;
  t.g = a;
  t.g.tm_w = b.map_gcnt_w;
  t.g.epi.r_hi = t.g.epi.r_lo = nullptr;  // gcn_residual rides in the GEMM as the fourth part
  memset(t.coef, 0, sizeof t.coef);
  t.n_parts = 4;
  const dim3 grid(persistent_grid(m, bt.n_tiles * a.n_frames)), block(384);
  const bool v25 = m->cfg.vertices == 25;
  if (bc.cout == 128 && bc.cin == 64) {
    if (v25) CK(launch_k(k_tc_agcnt<25, 1, 128>, grid, block, TcAgcntCfg<25, 1>::kSmemBytes, s, t));
    else CK(launch_k(k_tc_agcnt<18, 1, 128>, grid, block, TcAgcntCfg<18, 1>::kSmemBytes, s, t));
  } else if (bc.cout == 128) {
    if (v25) CK(launch_k(k_tc_agcnt<25, 2, 128>, grid, block, TcAgcntCfg<25, 2>::kSmemBytes, s, t));
    else CK(launch_k(k_tc_agcnt<18, 2, 128>, grid, block, TcAgcntCfg<18, 2>::kSmemBytes, s, t));
  } else {
    if (v25) CK(launch_k(k_tc_agcnt<25, 2, 256>, grid, block, TcAgcntCfg<25, 2>::kSmemBytes, s, t));
    else CK(launch_k(k_tc_agcnt<18, 2, 256>, grid, block, TcAgcntCfg<18, 2>::kSmemBytes, s, t));
  }
  return COSK_OK;
#endif
}

// Arguments of k_tc_tcn / k_tc_tcn2 for one frame.  n_taps = kTaps: the temporal conv of input n over the slots of frames
// n-8 .. n of the ring `x` (with phase timers); n_taps = 1: a token-major GEMM on slot 0 of `x`.  The residual rows are slot
// res_slot of `res` (nullptr: none), taken as kb_res extra K-blocks of the GEMM, or, with `res_epi`, added by the epilogue.
TcTcnArgs make_tc_tcn_args(const cosk_model *m, const Batch &bt, const ActBuf &x, int n_taps, long long n, int kb_per_tap,
                           const CUtensorMap &w, const float *bias, const ActBuf *res, int res_slot, int kb_res, bool res_epi,
                           const ActBuf &y, int y_slot) {
  TcTcnArgs a;
  a.tm_ring = x.map;
  a.tm_res = kb_res ? res->map : x.map;
  a.tm_w = w;
  for (int k = 0; k < kTaps; ++k) a.tap_row[k] = (int)x.row_hi(n_taps == 1 ? 0 : mod_slot(n - (kTaps - 1) + k, x.slots));
  a.res_row = res ? (int)res->row_hi(res_slot) : 0;
  a.t_alloc = (int)bt.t_alloc;
  a.n_taps = n_taps;
  a.kb_per_tap = kb_per_tap;
  a.kb_res = kb_res;
  a.n_tiles = bt.n_tiles;
  a.tile_tokens = bt.tile_tokens;
  a.reverse = n_taps == kTaps ? 1 : 0;
  a.n_tokens = bt.n_tokens;
  a.epi.bias = bias;
  a.epi.r_hi = res_epi ? res->hi(res_slot) : nullptr;
  a.epi.r_lo = res_epi ? res->lo(res_slot) : nullptr;
  a.epi.cs_r = res ? res->cs : 0;
  a.epi.y_hi = y.hi(y_slot);
  a.epi.y_lo = y.lo(y_slot);
  a.epi.cs_out = y.cs;
  a.trace = n_taps == kTaps ? m->d_trace : nullptr;
  a.dbg = m->d_dbg;
  return a;
}

// The 128- and 256-channel temporal convs run on CTA pairs (k_tc_tcn2) once there are two tiles to pair; the HBM-bound
// 64-channel ones stay on single CTAs.
bool tcn_on_pair(const Batch &bt, int width) { return bt.n_tiles >= 2 && (width == 128 || width == 256); }

// The temporal-conv kernel of output width `width` (64 / 128 / 256): the 9-tap conv of a block, or a plain token-major GEMM
// with one tap.  `half` is the weight map with half-height boxes the 256-wide pair kernel wants.
int launch_tcn(cosk_model *m, const Batch &bt, int width, TcTcnArgs &a, const CUtensorMap &half, cudaStream_t s) {
  if (tcn_on_pair(bt, width)) {
    // stacked-B width (128): CTA 0 loads the whole hi plane, CTA 1 the whole lo plane (full-height box);
    // C = 256: each CTA loads its half of the rows of both planes
    if (width > 128) a.tm_w = half;
    if (width == 128) return launch_tc_tcn2<128>(m, bt, a, s);
    return launch_tc_tcn2<256>(m, bt, a, s);
  }
  if (width == 64) return launch_tc_tcn<64>(m, bt, a, s);
  if (width == 128) return launch_tc_tcn<128>(m, bt, a, s);
  return launch_tc_tcn<256>(m, bt, a, s);
}

// Self-attention unit of CoS-TR (GcnUnitAttention, only_attention): qkv conv on the data_bn-normalised frame, 8-head
// attention over the vertices of each skeleton, then the output conv + bn + skip + ReLU -- the last one is the
// temporal-conv kernel run with a single tap on the attention rows.
int run_attention_unit(cosk_model *m, const Batch &bt, int i, const ActBuf &in, int in_slot, int ring_slot, cudaStream_t s) {
  const cosk_block_cfg &bc = m->cfg.blocks[i];
  BlockW &b = m->blk[i];
  const BlockBufs &buf = bt.blk[i];
  const GcnRoute g = b.route.gcn;
  const int dk = bc.cout / 4, dv = bc.cout, nq = 2 * dk + dv;
  int rc;
  if (g != GcnRoute::kSaSimt) {
    {  // data_bn of the unit as a pre-pass: the GEMM operand must exist in memory for TMA
      SaAffineArgs a;
      a.x_hi = in.hi(in_slot);
      a.x_lo = in.lo(in_slot);
      a.y_hi = buf.sa_x.hi(0);
      a.y_lo = buf.sa_x.lo(0);
      a.cs = in.cs;
      a.c = bc.cin;
      a.V = m->cfg.vertices;
      a.scale = b.d_sa_scale;
      a.shift = b.d_sa_shift;
      a.n_tokens = bt.n_tokens;
      const long long n = bt.n_tokens * (bc.cin / 8);
      CK(launch_k(k_sa_affine, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, s, a));
      m->launches++;
    }
    if (g == GcnRoute::kSaTcFused) {
      TcSaArgs a;
      a.tm_x = buf.sa_x.map;
      a.tm_w = b.map_sa_fw;
      a.x_row = (int)buf.sa_x.row_hi(0);
      a.t_alloc = (int)bt.t_alloc;
      a.cin = bc.cin;
      a.n_tiles = bt.n_tiles;
      a.tile_tokens = bt.tile_tokens;
      a.V = m->cfg.vertices;
      a.n_tokens = bt.n_tokens;
      a.bias = b.d_sa_fbias;
      a.y_hi = buf.sa.hi(0);
      a.y_lo = buf.sa.lo(0);
      a.cs_out = buf.sa.cs;
      a.dbg = m->d_dbg;
      const dim3 grid(persistent_grid(m, bt.n_tiles));
      if (bc.cout == 128) CK(launch_k(k_tc_sa<16>, grid, dim3(384), TcSaCfg<16>::kSmemBytes, s, a));
      else CK(launch_k(k_tc_sa<32>, grid, dim3(384), TcSaCfg<32>::kSmemBytes, s, a));
      m->launches++;
    } else {  // qkv conv = single-tap temporal-conv kernel without ReLU
      TcTcnArgs a = make_tc_tcn_args(m, bt, buf.sa_x, 1, 0, bc.cin / kBK, b.map_sa_q, b.d_sa_qbias, nullptr, 0, 0, false, buf.sa_q, 0);
      a.epi.floor = -INFINITY;
      if ((rc = launch_tcn(m, bt, kSaQkvCols, a, b.map_sa_q, s))) return rc;
      m->launches++;
    }
  } else {
    SaQkvArgs a;
    a.x_hi = in.hi(in_slot);
    a.x_lo = in.lo(in_slot);
    a.cs_in = in.cs;
    a.cin = bc.cin;
    a.in_scale = b.d_sa_scale;
    a.in_shift = b.d_sa_shift;
    a.w = b.d_sa_qkv_w;
    a.bias = b.d_sa_qkv_b;
    a.nq = nq;
    a.V = m->cfg.vertices;
    a.n_tokens = bt.n_tokens;
    a.tile_tokens = bt.tile_tokens;
    a.qkv = bt.d_qkv;
    dim3 grid(bt.n_tiles, (nq + kSimtN - 1) / kSimtN);
    CK(launch_k(k_sa_qkv, grid, dim3(256), 0, s, a));
    m->launches++;
  }
  if (g != GcnRoute::kSaTcFused) {
    SaAttnArgs a;
    a.qkv = bt.d_qkv;
    a.q_hi = g == GcnRoute::kSaTcQkv ? buf.sa_q.hi(0) : nullptr;
    a.q_lo = g == GcnRoute::kSaTcQkv ? buf.sa_q.lo(0) : nullptr;
    a.cs_q = buf.sa_q.cs;
    a.dk = dk;
    a.dv = dv;
    a.V = m->cfg.vertices;
    a.n_tokens = bt.n_tokens;
    a.tile_tokens = bt.tile_tokens;
    a.y_hi = buf.sa.hi(0);
    a.y_lo = buf.sa.lo(0);
    a.cs_out = buf.sa.cs;
    const int dvh = dv / kSaHeads;
    if (dvh == 8) CK(launch_k(k_sa_attn<8>, dim3(bt.n_tiles), dim3(256), 0, s, a));
    else if (dvh == 16) CK(launch_k(k_sa_attn<16>, dim3(bt.n_tiles), dim3(256), 0, s, a));
    else if (dvh == 32) CK(launch_k(k_sa_attn<32>, dim3(bt.n_tiles), dim3(256), 0, s, a));
    else CK(launch_k(k_sa_attn_any, dim3(bt.n_tiles), dim3(128), 0, s, a));
    m->launches++;
  }
  if ((rc = prof_mark(m, 1, i, s))) return rc;
  const bool skip = bc.cin == bc.cout;  // skip_conn and in_channels == out_channels (s_tr.py:464-467)
  if (b.route.sa_out_tc) {
    // the scaled skip connection is a K-block of the GEMM
    TcTcnArgs a = make_tc_tcn_args(m, bt, buf.sa, 1, 0, bc.cout / kBK, b.map_sa_w, b.d_gcn_b, &in, in_slot, skip ? bc.cin / kBK : 0, false,
                                   buf.ring, ring_slot);
    if ((rc = launch_tcn(m, bt, bc.cout, a, b.map_sa_w_half, s))) return rc;
  } else {
    TcnArgs a;
    for (int k = 0; k < kTaps; ++k) {
      a.tap_hi[k] = buf.sa.hi(0);
      a.tap_lo[k] = buf.sa.lo(0);
    }
    a.n_taps = 1;
    a.cs = buf.sa.cs;
    a.c = bc.cout;
    a.w = b.d_gcn_w;
    a.r_hi = in.hi(in_slot);
    a.r_lo = in.lo(in_slot);
    a.cs_r = in.cs;
    a.cr = bc.cin;
    a.res_kind = skip ? COSK_RES_CONV : COSK_RES_NONE;  // diag(skip scale) as a 1x1 "conv" on the input rows
    a.w_r = b.d_res_w_sa;
    a.bias = b.d_gcn_b;
    a.y_hi = buf.ring.hi(ring_slot);
    a.y_lo = buf.ring.lo(ring_slot);
    a.cs_out = buf.ring.cs;
    a.n_tokens = bt.n_tokens;
    a.tile_tokens = bt.tile_tokens;
    dim3 grid(bt.n_tiles, (bc.cout + kSimtN - 1) / kSimtN);
    CK(launch_k(k_tcn_simt, grid, dim3(256), 0, s, a));
  }
  m->launches++;
  return COSK_OK;
}

// Graph conv of block i for n_frames executions: frame f reads slot in_walk.slot(f) of `in` and writes slot ring_walk.slot(f)
// of the block's temporal ring.  Time-batched (n_frames > 1) only on the routes batched_ok admits.
int run_gcn(cosk_model *m, const Batch &bt, int i, const ActBuf &in, int n_frames, RingWalk in_walk, RingWalk ring_walk,
            cudaStream_t s) {
  const cosk_block_cfg &bc = m->cfg.blocks[i];
  BlockW &b = m->blk[i];
  const BlockBufs &buf = bt.blk[i];
  const Route &r = b.route;
  const int in_slot = in_walk.slot0, ring_slot = ring_walk.slot0;  // of the single-frame launches
  int rc = prof_mark(m, bc.gconv != COSK_GCONV_PLAIN ? 4 : 1, i, s);
  if (rc) return rc;
  if (bc.gconv == COSK_GCONV_ATTENTION) return run_attention_unit(m, bt, i, in, in_slot, ring_slot, s);
  if (r.attn == AttnRoute::kTc) {
    TcAttnArgs t;
    t.tm_x = in.map;
    t.tm_w = b.map_att_w;
    t.x_row = (int)in.row_hi(in_slot);
    t.t_alloc = (int)bt.t_alloc;
    t.cin = bc.cin;
    t.n_tiles = bt.n_tiles;
    t.tile_tokens = bt.tile_tokens;
    t.n_tokens = bt.n_tokens;
    t.bias = b.d_att_b;
    t.adj = b.d_adj;
    t.dense = bt.d_dense;
    t.dense_ld = 3 * bt.dense_vp;
    t.dbg = m->d_dbg;
    const int ic = bc.cout / 4;
    if (m->cfg.vertices == 25)
      rc = ic == 16   ? launch_tc_attn<16, 25>(m, bt, t, s)
           : ic == 32 ? launch_tc_attn<32, 25>(m, bt, t, s)
                      : launch_tc_attn<64, 25>(m, bt, t, s);
    else
      rc = ic == 16   ? launch_tc_attn<16, 18>(m, bt, t, s)
           : ic == 32 ? launch_tc_attn<32, 18>(m, bt, t, s)
                      : launch_tc_attn<64, 18>(m, bt, t, s);
    if (rc) return rc;
  } else if (r.attn == AttnRoute::kSmall) {
    // narrow first layer: embeddings computed per thread, same per-row softmax as the tensor-core kernel
    AttnSmallArgs t;
    t.x_hi = in.hi(in_slot);
    t.x_lo = in.lo(in_slot);
    t.cs_in = in.cs;
    t.cin = bc.cin;
    t.w = b.d_att_w;
    t.bias = b.d_att_b;
    t.adj = b.d_adj;
    t.n_tokens = bt.n_tokens;
    t.tile_tokens = bt.tile_tokens;
    t.dense = bt.d_dense;
    t.dense_ld = 3 * bt.dense_vp;
    if (m->cfg.vertices == 25) CK(launch_k(k_attn_small<16, 25>, dim3(bt.n_tiles), dim3(128), 0, s, t));
    else CK(launch_k(k_attn_small<16, 18>, dim3(bt.n_tiles), dim3(128), 0, s, t));
  } else if (r.attn == AttnRoute::kSimt) {
    // attention half: the per-token mixing rows of this frame go to the dense scratch
    AttnArgs t;
    t.x_hi = in.hi(in_slot);
    t.x_lo = in.lo(in_slot);
    t.cs_in = in.cs;
    t.cin = bc.cin;
    t.w = b.d_att_w;
    t.bias = b.d_att_b;
    t.inter_c = bc.cout / 4;
    t.adj = b.d_adj;
    t.V = m->cfg.vertices;
    t.n_tokens = bt.n_tokens;
    t.tile_tokens = bt.tile_tokens;
    t.dense = bt.d_dense;
    t.dense_ld = 3 * bt.dense_vp;
    t.dense_vp = bt.dense_vp;
    CK(launch_k(k_agcn_attn, dim3(bt.n_tiles), dim3(256), (size_t)2 * t.inter_c * kTileRows * sizeof(float), s, t));
  }
  if (r.attn != AttnRoute::kNone) {
    m->launches++;
    if ((rc = prof_mark(m, 1, i, s))) return rc;
  }
  const bool v25 = m->cfg.vertices == 25;
  const bool one_kb = bc.cin == kBK;  // one K-block per work item: single operand stage
  switch (r.gcn) {
    case GcnRoute::kTcAgcnt:
      rc = launch_tc_agcnt(m, bt, i, make_gcn_args(m, bt, i, in, n_frames, in_walk, ring_walk), s);
      break;
    case GcnRoute::kTcAgcn: {
      const TcGcnArgs a = make_gcn_args(m, bt, i, in, n_frames, in_walk, ring_walk);
      if (b.gcn_parts == 4) rc = v25 ? launch_tc_agcn<4, 1, 25>(m, bt, a, s) : launch_tc_agcn<4, 1, 18>(m, bt, a, s);
      else rc = v25 ? launch_tc_agcn<3, 2, 25>(m, bt, a, s) : launch_tc_agcn<3, 2, 18>(m, bt, a, s);
      break;
    }
    case GcnRoute::kTcT:
      rc = launch_tc_gcnt(m, bt, i, make_gcn_args(m, bt, i, in, n_frames, in_walk, ring_walk), s);
      break;
    case GcnRoute::kTc: {
      const TcGcnArgs a = make_gcn_args(m, bt, i, in, n_frames, in_walk, ring_walk);
      if (b.gcn_parts == 4) rc = one_kb ? launch_tc_gcn<4, 1>(m, bt, a, s) : launch_tc_gcn<4, 2>(m, bt, a, s);
      else rc = one_kb ? launch_tc_gcn<3, 1>(m, bt, a, s) : launch_tc_gcn<3, 2>(m, bt, a, s);
      break;
    }
    default: {  // kSimt, kSmall (time-batched: blockIdx.y = frame, pointers at slot 0 of their rings)
      const bool batched = n_frames > 1;
      const int res_conv = bc.cin != bc.cout ? 1 : 0;
      GcnArgs a;
      a.x_hi = in.hi(batched ? 0 : in_slot);
      a.x_lo = in.lo(batched ? 0 : in_slot);
      a.cs_in = in.cs;
      a.cin = bc.cin;
      a.y_hi = buf.ring.hi(batched ? 0 : ring_slot);
      a.y_lo = buf.ring.lo(batched ? 0 : ring_slot);
      a.cs_out = buf.ring.cs;
      a.cout = bc.cout;
      a.w = b.d_gcn_w;
      a.bias = b.d_gcn_b;
      a.res_conv = res_conv;
      a.res_identity = !res_conv;
      a.mix_ptr = b.d_mix_ptr;
      a.mix_src = b.d_mix_src;
      a.mix_val = b.d_mix_val;
      a.V = m->cfg.vertices;
      a.n_tokens = bt.n_tokens;
      a.tile_tokens = bt.tile_tokens;
      a.dense = bc.gconv == COSK_GCONV_ADAPTIVE ? bt.d_dense : nullptr;
      a.dense_ld = 3 * bt.dense_vp;
      a.dense_vp = bt.dense_vp;
      if (batched) {
        a.in_walk = in_walk;
        a.out_walk = ring_walk;
        a.in_slot_elems = in.slot_elems();
        a.out_slot_elems = buf.ring.slot_elems();
      }
      const int K = (3 + res_conv) * bc.cin;
      if (r.gcn == GcnRoute::kSmall)
        CK(launch_k(k_gcn_small, dim3(bt.n_tiles, n_frames), dim3(256), (size_t)(K + 1) * bc.cout * sizeof(float), s, a));
      else
        CK(launch_k(k_gcn_simt, dim3(bt.n_tiles, (bc.cout + kSimtN - 1) / kSimtN), dim3(256), 0, s, a));
    }
  }
  if (rc) return rc;
  m->launches++;
  return COSK_OK;
}

// Temporal conv of block i for n_frames firing executions, the first on input n: frame f adds the delayed residual from slot
// res_walk.slot(f) of `in` and writes slot out_walk.slot(f) of the block's output ring (time-batched: tensor cores only).
int run_tcn(cosk_model *m, const Batch &bt, int i, const ActBuf &in, long long n, int n_frames, RingWalk res_walk, RingWalk out_walk,
            cudaStream_t s) {
  const cosk_block_cfg &bc = m->cfg.blocks[i];
  BlockW &b = m->blk[i];
  const BlockBufs &buf = bt.blk[i];
  int rc = prof_mark(m, 2, i, s);
  if (rc) return rc;
  if (b.route.tcn_tc) {
    const bool batched = n_frames > 1;  // pointers at slot 0 of their rings, the slots from the walks
    const bool kblock = tcn_res_kblock(bc);
    TcTcnArgs a = make_tc_tcn_args(m, bt, buf.ring, kTaps, n, bc.cout / kBK, b.map_tcn_w, b.d_tcn_b, &in, batched ? 0 : res_walk.slot0,
                                   kblock ? bc.cin / kBK : 0, bc.res_kind == COSK_RES_IDENTITY && !kblock, buf.out,
                                   batched ? 0 : out_walk.slot0);
    if (batched) {
      a.n_frames = n_frames;
      a.slot_rows = (int)(2 * bt.t_alloc);
      a.tap_walk = ring_walk(n - (kTaps - 1), bc.stride, bt.R);
      a.res_walk = res_walk;
      a.out_walk = out_walk;
      a.out_slot_elems = buf.out.slot_elems();
      a.res_slot_elems = in.slot_elems();
    }
    if ((rc = launch_tcn(m, bt, bc.cout, a, b.map_tcn_w_half, s))) return rc;
  } else {
    TcnArgs a;
    for (int k = 0; k < kTaps; ++k) {
      const int slot = mod_slot(n - (kTaps - 1) + k, bt.R);  // frame n-8+k
      a.tap_hi[k] = buf.ring.hi(slot);
      a.tap_lo[k] = buf.ring.lo(slot);
    }
    a.n_taps = kTaps;
    a.cs = buf.ring.cs;
    a.c = bc.cout;
    a.w = b.d_tcn_w;
    a.r_hi = in.hi(res_walk.slot0);
    a.r_lo = in.lo(res_walk.slot0);
    a.cs_r = in.cs;
    a.cr = bc.cin;
    a.res_kind = bc.res_kind;
    a.w_r = b.d_res_w;
    a.bias = b.d_tcn_b;
    a.y_hi = buf.out.hi(out_walk.slot0);
    a.y_lo = buf.out.lo(out_walk.slot0);
    a.cs_out = buf.out.cs;
    a.n_tokens = bt.n_tokens;
    a.tile_tokens = bt.tile_tokens;
    dim3 grid(bt.n_tiles, (bc.cout + kSimtN - 1) / kSimtN);
    CK(launch_k(k_tcn_simt, grid, dim3(256), 0, s, a));
  }
  m->launches++;
  return COSK_OK;
}

// Graph conv + temporal conv of a 64 -> 64 block as one launch (k_tc_block64).  `fire`: the temporal conv emits on this step.
int run_block64(cosk_model *m, const Batch &bt, int i, const ActBuf &in, int in_slot, long long n, bool fire, int res_slot, int out_slot,
                cudaStream_t s) {
  BlockW &b = m->blk[i];
  const BlockBufs &buf = bt.blk[i];
  int rc = prof_mark(m, 5, i, s);
  if (rc) return rc;
  TcBlockArgs a;
  a.tm_x = in.map;
  a.tm_ring = buf.ring.map;
  a.tm_gw = b.map_gcnp_w;
  a.tm_tw = b.map_tcn_w_full;
  a.n_parts = b.gcnp_parts;
  a.x_row = (int)in.row_hi(in_slot);
  a.res_row = fire ? (int)in.row_hi(res_slot) : 0;
  for (int k = 0; k < kTaps - 1; ++k) a.tap_row[k] = (int)buf.ring.row_hi(mod_slot(n - (kTaps - 1) + k, bt.R));  // frame n-8+k
  a.t_alloc = (int)bt.t_alloc;
  a.with_tcn = fire ? 1 : 0;
  a.V = m->cfg.vertices;
  a.n_tiles = bt.n_tiles;
  a.tile_tokens = bt.tile_tokens;
  a.n_tokens = bt.n_tokens;
  a.mix_ptr = b.d_mix_ptr;
  a.mix_src = b.d_mix_src;
  a.mix_val = b.d_mix_val;
  a.gbias = b.d_gcn_b;
  const int ring_slot = (int)(n % bt.R);
  a.g_hi = buf.ring.hi(ring_slot);
  a.g_lo = buf.ring.lo(ring_slot);
  a.cs_g = buf.ring.cs;
  a.tepi.bias = b.d_tcn_b;
  a.tepi.r_hi = nullptr;  // the delayed identity residual is a K-block of the temporal GEMM
  a.tepi.r_lo = nullptr;
  a.tepi.cs_r = 0;
  a.tepi.y_hi = buf.out.hi(out_slot);
  a.tepi.y_lo = buf.out.lo(out_slot);
  a.tepi.cs_out = buf.out.cs;
  a.trace = m->d_trace;
  a.dbg = m->d_dbg;
  CK(launch_k(k_tc_block64, dim3(persistent_grid(m, bt.n_tiles)), dim3(512), TcBlockCfg::kSmemBytes, s, a));
  m->launches++;
  return COSK_OK;
}

// k_input: n_frames input frames (frame f at x + f * x_frame_stride) -> slots walk.slot(f) of the input ring, data_bn folded in
int run_input(cosk_model *m, const Batch &bt, const float *x, long long nc_stride, long long x_frame_stride, int n_frames,
              RingWalk walk, cudaStream_t s) {
  const cosk_config &c = m->cfg;
  const long long total = bt.n_tokens * bt.xin.cs;
  const int threads = 256;
  const long long blocks = (total + threads - 1) / threads;
  CK(launch_k(k_input, dim3((unsigned)blocks, (unsigned)n_frames), dim3(threads), 0, s, x, nc_stride, c.c_in, c.vertices, c.persons,
              (const float *)(c.data_bn ? m->d_bn_scale : nullptr), (const float *)(c.data_bn ? m->d_bn_shift : nullptr), bt.xin.hi(0),
              bt.xin.lo(0), bt.xin.cs, bt.n_tokens, x_frame_stride, walk, bt.xin.slot_elems()));
  m->launches++;
  return COSK_OK;
}

// k_head over n_frames emissions of the last block, frame f from slot in_walk.slot(f) of its output ring (`zero`: one zero
// vector enters the pooling window instead).  One frame emits logits iff `emit`; more emit from frame first_emit on,
// emission j at out + j * out_stride.
int run_head(cosk_model *m, Batch &bt, int n_frames, RingWalk in_walk, bool zero, int emit, int first_emit, float *out,
             long long out_stride, cudaStream_t s) {
  const cosk_config &c = m->cfg;
  const ActBuf &y = bt.blk[c.n_blocks - 1].out;
  const bool batched = n_frames > 1;  // y_* at slot 0 of the ring, the slots from the walk
  int rc = prof_mark(m, 3, -1, s);
  if (rc) return rc;
  HeadArgs h;
  h.y_hi = zero ? nullptr : y.hi(batched ? 0 : in_walk.slot0);
  h.y_lo = zero ? nullptr : y.lo(batched ? 0 : in_walk.slot0);
  h.cs = y.cs;
  h.c = y.c;
  h.V = c.vertices;
  h.S = c.persons;
  h.ring = bt.d_pool_ring;
  h.sum = bt.d_pool_sum;
  h.slot = (int)(bt.cnt.pool_n % c.pool_size);
  h.P = c.pool_size;
  h.n_streams = bt.n_streams;
  h.emit = emit;
  h.w = m->d_fc_w;
  h.b = m->d_fc_b;
  h.classes = c.classes;
  h.out = out;
  h.first_emit = first_emit;
  h.out_stride = out_stride;
  if (batched) {
    h.n_frames = n_frames;
    h.in_walk = in_walk;
    h.in_slot_elems = y.slot_elems();
  }
  CK(launch_k(k_head, dim3((unsigned)((bt.n_streams + kHeadStreams - 1) / kHeadStreams)), dim3(256 * kHeadStreams),
              (size_t)kHeadStreams * (2 * y.cs + y.c) * sizeof(float), s, h));
  m->launches++;
  bt.cnt.pool_n += n_frames;
  return COSK_OK;
}

// k_read_block: slot `slot` of a block's output ring -> fp32 at dst
int read_block(cosk_model *m, const Batch &bt, const ActBuf &o, int slot, float *dst, cudaStream_t s) {
  const long long total = bt.n_tokens * o.c;
  CK(launch_k(k_read_block, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, s, (const __nv_bfloat16 *)o.hi(slot),
              (const __nv_bfloat16 *)o.lo(slot), o.cs, o.c, m->cfg.vertices, bt.n_tokens, dst));
  m->launches++;
  return COSK_OK;
}

// ---- the integer schedule: one firing rule for the walk, cosk_simulate_schedule and cosk_schedule_compatible ----------
// co.Conv2d step semantics: the n-th input (0-based) of a 9-tap temporal conv with padding p and stride s produces an output
// iff n >= 8 - p and (n - (8 - p)) % s == 0   (SURVEY.md section 3.3).  Among the inputs n0 .. n0+F-1 of such a conv,
// `first` is the first firing input at or after n0 (it may lie past the range) and `count` how many of them fire.
struct Firing {
  long long first, count;
};
Firing firing(int padding, int stride, long long n0, long long F) {
  const int p0 = (kTaps - 1) - padding;  // first firing input of the stream
  const long long nf = n0 < p0 ? p0 : n0 + ((p0 - n0) % stride + stride) % stride;
  return {nf, nf <= n0 + F - 1 ? (n0 + F - 1 - nf) / stride + 1 : 0};
}
// co.AvgPool1d(P, stride 1, padding pp): the m-th pooled vector yields logits iff m >= P - 1 - pp.  Of F vectors entering the
// window from the pool_n-th on, how many come before the first logits.
long long head_skip(const cosk_config &c, long long pool_n, long long F) {
  return std::min(std::max((long long)c.pool_size - 1 - c.pool_padding - pool_n, 0LL), F);
}

// One frame of the emission bookkeeping: advances n_in and pool_n of `k`, writes n_blocks + 1 flags laid out like
// cosk_last_schedule.
void schedule_frame(const cosk_config &c, Counters &k, int32_t *flags) {
  bool alive = true;
  for (int i = 0; i < c.n_blocks; ++i) {
    flags[i] = 0;
    if (!alive) continue;
    alive = firing(c.padding, c.blocks[i].stride, k.n_in[i]++, 1).count > 0;
    flags[i] = alive ? 1 : 0;
  }
  int emit = 0;
  if (alive) emit = c.classes > 0 ? head_skip(c, k.pool_n++, 1) == 0 : 1;
  flags[c.n_blocks] = emit;
}

// The counters the walk (and schedule_frame) reaches after `frames` frames from zero.
Counters counters_at(const cosk_config &c, long long frames) {
  Counters k;
  k.frame = frames;
  long long n = frames;
  for (int i = 0; i < c.n_blocks; ++i) {
    k.n_in[i] = n;
    n = k.n_out[i] = firing(c.padding, c.blocks[i].stride, 0, n).count;
  }
  k.pool_n = c.classes > 0 ? n : 0;
  return k;
}

// Every block has reached its first firing input and the pooling window its first emission: the schedule is periodic.
bool past_warmup(const cosk_config &c, const Counters &k) {
  for (int i = 0; i < c.n_blocks; ++i)
    if (k.n_in[i] < firing(c.padding, c.blocks[i].stride, 0, 0).first) return false;
  return c.classes <= 0 || head_skip(c, k.pool_n, 1) == 0;
}

// ---- the walk over the stack (cosk_step, cosk_steps) ---------------------------------------------------------------
// Time-batched chunks (cosk_steps with a time chunk > 1) are available when every block runs on the tensor-core CoST-GCN
// kernels (k_tc_gcn or k_tc_gcnt, k_gcn_small for the first layer, k_tc_tcn / k_tc_tcn2).
bool batched_ok(const cosk_model *m, const Batch &bt) {
  if (bt.tchunk <= 1 || m->d_trace) return false;
  for (const BlockW &b : m->blk) {
    const Route &r = b.route;
    if (r.attn != AttnRoute::kNone || !r.tcn_tc) return false;
    if (r.gcn != GcnRoute::kTc && r.gcn != GcnRoute::kTcT && r.gcn != GcnRoute::kSmall) return false;
  }
  return true;
}

// F0 input frames (frame f at x + f * x_frame_stride) enter the stack, which is walked module by module: every block runs
// over the F executions its predecessor emitted, one launch per kernel; the work items of a launch are (frame, tile) pairs
// and every frame's ring slots follow from a RingWalk.  Emission j of the head (or of a headless stack's last block) is
// written at out + (*cnt + j) * out_stride, and *cnt advances; once max_out are stored, later ones land in the last slot.
//
// `frame_by_frame` (F0 == 1): a block routed to k_tc_block64 runs as that one kernel.  Time-batched chunks run it as graph
// conv + temporal conv launches, a chunk of one frame too: frame n's temporal conv reads the graph-conv outputs of frames
// n-8 .. n-1, which a launch covering many frames would produce concurrently, and the one kernel rounds differently.
//
// End-of-sequence flush (`flush` >= 0; forward_steps(pad_end=True) of the library: every temporal module is fed its own end
// padding once the clip is over, module by module): no input.  `flush` = i in [0, n_blocks) pushes one ZERO frame into the
// temporal conv of block i (not through its graph conv: co.forward_stepping modules have no padding), `flush` = n_blocks
// pushes one zero vector into the pooling window; whatever that emits propagates through the later stages like a regular
// frame.  The frame counter does not advance.
int walk(cosk_model *m, Batch &bt, const float *x, long long nc_stride, long long x_frame_stride, int F0, bool frame_by_frame,
         float *out, long long out_stride, int32_t max_out, int32_t *cnt, cudaStream_t s, int flush = -1) {
  const cosk_config &c = m->cfg;
  Counters &k = bt.cnt;
  int rc;
  if ((rc = prof_mark(m, 0, -1, s))) return rc;
  if (flush < 0 && (rc = run_input(m, bt, x, nc_stride, x_frame_stride, F0, ring_walk(k.frame, 1, bt.Ro), s))) return rc;
  const ActBuf *in = &bt.xin;
  int F = flush < 0 ? F0 : 0;  // executions of the current block in this walk == emissions of its predecessor
  for (int i = 0; i < c.n_blocks; ++i) {
    const Route &route = m->blk[i].route;
    const BlockBufs &buf = bt.blk[i];
    const cosk_block_cfg &bc = c.blocks[i];
    const bool zero_in = i == flush;  // the zero frame enters this block's temporal conv directly
    if (zero_in) F = 1;
    bt.last_flags[i] = 0;
    if (F == 0) {
      in = &buf.out;
      continue;
    }
    const long long n0 = k.n_in[i];  // index of the first execution == index of the predecessor's emission
    const Firing fire = firing(c.padding, bc.stride, n0, F);
    const int F_out = (int)fire.count;
    const bool fused = frame_by_frame && route.block64 && in->has_map && !zero_in;
    if (zero_in) {
      const int rs = (int)(n0 % bt.R);
      CK(cudaMemsetAsync(buf.ring.hi(rs), 0, (size_t)2 * buf.ring.t_alloc * buf.ring.cs * sizeof(__nv_bfloat16), s));
    } else if (fused) {
      const int res_slot = F_out > 0 ? (int)((n0 - kResDelay) % bt.Ro) : 0;
      if ((rc = run_block64(m, bt, i, *in, (int)(n0 % bt.Ro), n0, F_out > 0, res_slot, (int)(k.n_out[i] % bt.Ro), s))) return rc;
    } else if ((rc = run_gcn(m, bt, i, *in, F, ring_walk(n0, 1, bt.Ro), ring_walk(n0, 1, bt.R), s))) {
      return rc;
    }
    if (F_out > 0 && !fused &&
        (rc = run_tcn(m, bt, i, *in, fire.first, F_out, ring_walk(fire.first - kResDelay, bc.stride, bt.Ro),
                      ring_walk(k.n_out[i], 1, bt.Ro), s)))
      return rc;
    // did the block fire on its last execution?  (schedule parity is defined per frame)
    bt.last_flags[i] = (F_out > 0 && fire.first + (long long)(F_out - 1) * bc.stride == n0 + F - 1) ? 1 : 0;
    k.n_in[i] += F;
    k.n_out[i] += F_out;
    F = F_out;
    in = &buf.out;
  }
  // head over the F emissions of the last block; a flushed zero vector enters the pooling window alone (a stack without a
  // head has no window to flush)
  const bool head_zero = flush == c.n_blocks;
  if (head_zero) F = c.classes > 0 ? 1 : 0;
  int emit_last = 0;
  if (F > 0) {
    const long long o0 = k.n_out[c.n_blocks - 1] - F;  // index of the first of these emissions
    if (c.classes > 0) {
      const int skip = (int)head_skip(c, k.pool_n, F);  // frames before the first logits
      const int n_emit = F - skip;
      const int32_t room = *cnt < max_out ? max_out - *cnt : 0;
      float *dst = out + (long long)(*cnt < max_out ? *cnt : max_out - 1) * out_stride;
      // more emissions than room: they all land in the last slot
      if ((rc = run_head(m, bt, F, ring_walk(o0, 1, bt.Ro), head_zero, F == 1 ? n_emit : 0, skip, dst,
                         n_emit <= room ? out_stride : 0, s)))
        return rc;
      *cnt += n_emit;
      emit_last = n_emit > 0 ? 1 : 0;
    } else {
      for (int f = 0; f < F; ++f) {
        float *dst = out + (long long)(*cnt < max_out ? *cnt : max_out - 1) * out_stride;
        if ((rc = read_block(m, bt, bt.blk[c.n_blocks - 1].out, mod_slot(o0 + f, bt.Ro), dst, s))) return rc;
        *cnt += 1;
      }
      emit_last = 1;
    }
  }
  if ((rc = prof_mark(m, -1, -1, s))) return rc;  // closes the last interval of this walk
  bt.last_flags[c.n_blocks] = (emit_last && bt.last_flags[c.n_blocks - 1]) ? 1 : 0;
  if (flush < 0) k.frame += F0;
  return COSK_OK;
}

// The end of a stepping call's walks.  A walk that stopped half way leaves the counters partly advanced: the failure latch
// refuses further steps.  Otherwise, if anything emitted, the watchdog word is copied to pinned memory behind the call's
// kernels, without a host sync, for step_entry of the next call to look at.  The device word only goes from 0 to a code
// until a reset, so one copy per call sees what a copy behind every emitting frame would.
int end_walks(cosk_model *m, int rc, int32_t cnt, cudaStream_t s) {
  if (!rc && cnt > 0 && m->h_dbg &&
      cudaMemcpyAsync(m->h_dbg, m->d_dbg, sizeof(unsigned int), cudaMemcpyDeviceToHost, s) != cudaSuccess)
    rc = fail(m, COSK_ERR_CUDA, "cudaMemcpyAsync of the watchdog word failed");
  if (rc) m->failed = true;
  return rc;
}

// F frames of a (N, C, T, V, S) clip through the stack, the first at x (nc_stride = T*V*S): chunks of the time chunk where
// batched_ok admits them, else frame by frame (cosk_steps, cosk_prime_streams).
int walk_frames(cosk_model *m, Batch &bt, const float *x, long long nc_stride, int F, float *out, long long out_stride,
                int32_t max_out, int32_t *cnt, cudaStream_t s) {
  const long long frame_elems = (long long)m->cfg.vertices * m->cfg.persons;
  const bool batched = batched_ok(m, bt);
  const int chunk = batched ? bt.tchunk : 1;
  int rc = COSK_OK;
  for (int t0 = 0; t0 < F && !rc; t0 += chunk)
    rc = walk(m, bt, x + t0 * frame_elems, nc_stride, frame_elems, std::min(chunk, F - t0), !batched, out, out_stride, max_out, cnt, s);
  return rc;
}

// cosk_describe's name of the kernels that serve a block's graph conv (the adaptive one: attention half + mix)
std::string gcn_name(const BlockW &b) {
  static const char *const attn[] = {"", "k_agcn_attn+", "k_attn_small+", "k_tc_attn+"};  // by AttnRoute
  char t[64] = "";
  switch (b.route.gcn) {
    case GcnRoute::kSimt: snprintf(t, sizeof t, "k_gcn_simt"); break;
    case GcnRoute::kSmall: snprintf(t, sizeof t, "k_gcn_small"); break;
    case GcnRoute::kTc: snprintf(t, sizeof t, "k_tc_gcn<%d> GEMM-then-mix", b.gcn_parts); break;
    case GcnRoute::kTcT: snprintf(t, sizeof t, "k_tc_gcnt<%d> channel-major, mix in registers", b.gcnt_parts); break;
    case GcnRoute::kTcAgcn: snprintf(t, sizeof t, "k_tc_agcn"); break;
    case GcnRoute::kTcAgcnt: snprintf(t, sizeof t, "k_tc_agcnt"); break;
    case GcnRoute::kSaSimt: snprintf(t, sizeof t, "k_sa_qkv+k_sa_attn"); break;
    case GcnRoute::kSaTcQkv: snprintf(t, sizeof t, "k_tc_tcn(qkv)+k_sa_attn"); break;
    case GcnRoute::kSaTcFused: snprintf(t, sizeof t, "k_tc_sa"); break;
  }
  return std::string(attn[(int)b.route.attn]) + t;
}

// The geometry and ring sizes of `n_streams` streams at time chunk `time_chunk` into `b`, which holds no buffers; nothing
// is allocated.  Refuses a time chunk out of range and a batch whose rings need more than 32-bit rows (`b` left empty).
int batch_geometry(cosk_model *m, int64_t n_streams, int time_chunk, Batch &b) {
  const cosk_config &c = m->cfg;
  if (n_streams < 1 || time_chunk < 1 || time_chunk > 4096)
    return fail(m, COSK_ERR_ARG, "%lld streams at time chunk %d", (long long)n_streams, time_chunk);
  b.n_streams = n_streams;
  b.tchunk = time_chunk;
  b.R = (kRingSlots - 1) + time_chunk;
  b.Ro = (kOutSlots - 1) + time_chunk;
  const long long skel = n_streams * c.persons;
  b.n_tokens = skel * c.vertices;
  b.skel_per_tile = kTileRows / c.vertices;
  b.tile_tokens = b.skel_per_tile * c.vertices;
  const long long n_tiles = (skel + b.skel_per_tile - 1) / b.skel_per_tile;
  // +1 tile: with an odd tile count the second CTA of the last pair walks a phantom tile (loads only)
  b.t_alloc = ((n_tiles + 1) * b.tile_tokens + (kTileRows - b.tile_tokens) + 7) / 8 * 8;
  if ((long long)b.R * 2 * b.t_alloc > 0x7fffffffLL) {
    b = Batch();
    return fail(m, COSK_ERR_ARG, "too many streams (x time chunk) for 32-bit rows");
  }
  b.n_tiles = (int)n_tiles;
  return COSK_OK;
}

int alloc_buffers(cosk_model *m, Batch &b) {
  const cosk_config &c = m->cfg;
  int rc = alloc_act(m, b, b.xin, b.Ro, c.c_in);
  if (rc) return rc;
  for (int i = 0; i < c.n_blocks; ++i) {
    if ((rc = alloc_act(m, b, b.blk[i].ring, b.R, c.blocks[i].cout))) return rc;
    if ((rc = alloc_act(m, b, b.blk[i].out, b.Ro, c.blocks[i].cout))) return rc;
  }
  if (c.classes > 0) {
    const size_t cl = (size_t)c.blocks[c.n_blocks - 1].cout;
    CK(cudaMalloc(&b.d_pool_ring, (size_t)c.pool_size * b.n_streams * cl * sizeof(float)));
    CK(cudaMalloc(&b.d_pool_sum, (size_t)b.n_streams * cl * sizeof(double)));
    b.state_bytes += (int64_t)((size_t)c.pool_size * b.n_streams * cl * sizeof(float) + (size_t)b.n_streams * cl * sizeof(double));
  }
  bool any_adaptive = false;
  int max_nq = 0;
  for (int i = 0; i < c.n_blocks; ++i) {
    any_adaptive |= c.blocks[i].gconv == COSK_GCONV_ADAPTIVE;
    if (c.blocks[i].gconv == COSK_GCONV_ATTENTION) {
      BlockBufs &buf = b.blk[i];
      max_nq = std::max(max_nq, 2 * (c.blocks[i].cout / 4) + c.blocks[i].cout);
      if ((rc = alloc_act(m, b, buf.sa, 1, c.blocks[i].cout))) return rc;
      CK(cudaMemset(buf.sa.ptr, 0, buf.sa.bytes()));
      const GcnRoute g = m->blk[i].route.gcn;
      if (g != GcnRoute::kSaSimt) {
        if ((rc = alloc_act(m, b, buf.sa_x, 1, c.blocks[i].cin))) return rc;
        CK(cudaMemset(buf.sa_x.ptr, 0, buf.sa_x.bytes()));
        if (g == GcnRoute::kSaTcQkv) {
          if ((rc = alloc_act(m, b, buf.sa_q, 1, kSaQkvCols))) return rc;
          CK(cudaMemset(buf.sa_q.ptr, 0, buf.sa_q.bytes()));
        }
      }
    }
  }
  if (max_nq) {
    const size_t bytes = (size_t)b.t_alloc * max_nq * sizeof(float);
    CK(cudaMalloc(&b.d_qkv, bytes));
    b.state_bytes += (int64_t)bytes;  // scratch, counted in the footprint
  }
  if (any_adaptive) {
    b.dense_vp = round_up(c.vertices, 4);
    const size_t bytes = (size_t)b.t_alloc * 3 * b.dense_vp * sizeof(float);
    CK(cudaMalloc(&b.d_dense, bytes));
    CK(cudaMemset(b.d_dense, 0, bytes));
    b.state_bytes += (int64_t)bytes;  // scratch, not state, but part of the per-stream footprint
  }
  CK(cudaMalloc(&b.d_idx, (size_t)b.n_streams * sizeof(long long)));  // index list of the per-stream calls, not counted
  return COSK_OK;
}

// Builds the batch of `n_streams` streams at time chunk `time_chunk` into `b`, which holds no buffers: counters zero,
// buffer contents undefined except the scratch, which starts zeroed.  Refusals (batch_geometry) come before any
// allocation; on failure `b` is left empty.
int alloc_batch(cosk_model *m, int64_t n_streams, int time_chunk, Batch &b) {
  int rc = batch_geometry(m, n_streams, time_chunk, b);
  if (!rc && (rc = alloc_buffers(m, b))) free_batch(b);
  return rc;
}

}  // namespace

#include "stream_state_host.cuh"

extern "C" {

const char *cosk_version(void) { return "cosk 0.1 (sm_100a)"; }

const char *cosk_last_error(const cosk_model *m) { return m ? m->err.c_str() : "null handle"; }

int cosk_create(const cosk_config *cfg, cosk_model **out) {
  if (!cfg || !out) return COSK_ERR_ARG;
  *out = nullptr;
  if (cfg->abi_version != COSK_ABI_VERSION) return COSK_ERR_ARG;
  if (cfg->n_blocks < 1 || cfg->n_blocks > COSK_MAX_BLOCKS) return COSK_ERR_ARG;
  if (cfg->vertices < 1 || cfg->vertices > kTileRows || cfg->persons < 1 || cfg->c_in < 1) return COSK_ERR_ARG;
  if (cfg->padding != 0 && cfg->padding != 4) return COSK_ERR_ARG;
  if (cfg->classes > 0 && (cfg->pool_size < 1 || cfg->pool_padding < 0 || cfg->pool_padding >= cfg->pool_size))
    return COSK_ERR_ARG;
  int prev = cfg->c_in;
  for (int i = 0; i < cfg->n_blocks; ++i) {
    const cosk_block_cfg &b = cfg->blocks[i];
    if (b.cin != prev || b.cout < 1 || (b.stride != 1 && b.stride != 2)) return COSK_ERR_ARG;
    if (b.res_kind == COSK_RES_IDENTITY && (b.cin != b.cout || b.stride != 1)) return COSK_ERR_ARG;
    if (b.res_kind < 0 || b.res_kind > 2) return COSK_ERR_ARG;
    if (b.gconv < COSK_GCONV_PLAIN || b.gconv > COSK_GCONV_ATTENTION) return COSK_ERR_ARG;
    if (b.gconv != COSK_GCONV_PLAIN && cfg->vertices > kAttnMaxV) return COSK_ERR_ARG;
    if (b.gconv == COSK_GCONV_ADAPTIVE && (b.cout < 4 || b.cout / 4 > kAttnMaxInter)) return COSK_ERR_ARG;
    // 8 heads over dk = cout/4 and dv = cout channels (models/s_tr/s_tr.py:72-78), head widths the kernel holds in registers
    if (b.gconv == COSK_GCONV_ATTENTION && (b.cout % 32 != 0 || b.cout / 32 > kSaMaxDkh || b.cout / 8 > kSaMaxDvh)) return COSK_ERR_ARG;
    prev = b.cout;
  }
  cosk_model *m = new cosk_model();
  m->cfg = *cfg;
  m->blk.resize(cfg->n_blocks);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || cfg->device < 0 || cfg->device >= ndev) {
    delete m;
    return COSK_ERR_CUDA;  // no CPU fallback: the library is useless without a CUDA device
  }
  DeviceGuard guard_(cfg->device);
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, cfg->device);
  m->num_sms = prop.multiProcessorCount;
  if (const char *e = getenv("COSK_FUSE_BLOCK")) m->fuse_block = atoi(e);
  if (const char *e = getenv("COSK_GCN_T")) m->gcn_transposed = atoi(e);
  if (const char *e = getenv("COSK_AGCN_T")) m->agcn_transposed = atoi(e);
  if (const char *e = getenv("COSK_TRACE")) {
    if (atoi(e) && cudaMalloc(&m->d_trace, 64 * sizeof(unsigned long long)) == cudaSuccess)
      cudaMemset(m->d_trace, 0, 64 * sizeof(unsigned long long));
  }
  const bool sm100 = prop.major == 10;
  if (!sm100 && cfg->path == COSK_PATH_AUTO) {
    delete m;
    return COSK_ERR_UNSUPPORTED;  // the tcgen05 kernels are sm_100a only
  }
  void *fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || fn == nullptr) {
    delete m;
    return COSK_ERR_CUDA;
  }
  m->encode = reinterpret_cast<EncodeTiledFn>(fn);
  if (cudaMalloc(&m->d_dbg, 4 * sizeof(unsigned int)) != cudaSuccess) {
    delete m;
    return COSK_ERR_CUDA;
  }
  cudaMemset(m->d_dbg, 0, 4 * sizeof(unsigned int));
  if (cudaHostAlloc(&m->h_dbg, 4 * sizeof(unsigned int), cudaHostAllocDefault) != cudaSuccess) {
    cudaFree(m->d_dbg);
    delete m;
    return COSK_ERR_CUDA;
  }
  memset(m->h_dbg, 0, 4 * sizeof(unsigned int));
  if (sm100 && set_smem_attrs(m) != COSK_OK) {
    fprintf(stderr, "cosk_create: %s\n", m->err.c_str());
    cudaFree(m->d_dbg);
    cudaFreeHost(m->h_dbg);
    delete m;
    return COSK_ERR_CUDA;
  }
  *out = m;
  return COSK_OK;
}

void cosk_destroy(cosk_model *m) {
  if (!m) return;
  DeviceGuard guard_(m->cfg.device);
  free_batch(m->batch);
  for (auto &b : m->blk) {
    dfree(b.d_gcn_w);
    dfree(b.d_gcn_b);
    dfree(b.d_tcn_w);
    dfree(b.d_res_w);
    dfree(b.d_tcn_b);
    dfree(b.d_mix_ptr);
    dfree(b.d_mix_src);
    dfree(b.d_mix_val);
    dfree(b.d_att_w);
    dfree(b.d_att_b);
    dfree(b.d_adj);
    dfree(b.d_gcn_w16);
    dfree(b.d_gcnp_w16);
    dfree(b.d_gcnt_w16);
    dfree(b.d_tcn_w16);
    dfree(b.d_att_w16);
    dfree(b.d_sa_scale);
    dfree(b.d_sa_shift);
    dfree(b.d_sa_qkv_w);
    dfree(b.d_sa_qkv_b);
    dfree(b.d_sa_w16);
    dfree(b.d_res_w_sa);
    dfree(b.d_sa_fw16);
    dfree(b.d_sa_fbias);
    dfree(b.d_sa_qw16);
    dfree(b.d_sa_qbias);
  }
  dfree(m->d_bn_scale);
  dfree(m->d_bn_shift);
  dfree(m->d_fc_w);
  dfree(m->d_fc_b);
  dfree(m->d_dbg);
  if (m->h_dbg) cudaFreeHost(m->h_dbg);
  dfree(m->d_trace);
  for (auto e : m->ev_pool) cudaEventDestroy(e);
  if (m->ev_idx) cudaEventDestroy(m->ev_idx);
  delete m;
}

int cosk_load_weights(cosk_model *m, const char *name, const float *host, size_t n) {
  if (!m || !name || !host) return COSK_ERR_ARG;
  std::vector<float> v(host, host + n);
  std::string s(name);
  m->prepared = false;
  if (s == "data_bn.scale") m->h_bn_scale = v;
  else if (s == "data_bn.shift") m->h_bn_shift = v;
  else if (s == "fc.w") m->h_fc_w = v;
  else if (s == "fc.b") m->h_fc_b = v;
  else if (s.rfind("block", 0) == 0) {
    size_t dot = s.find('.');
    if (dot == std::string::npos) return fail(m, COSK_ERR_ARG, "bad tensor name %s", name);
    int i = atoi(s.substr(5, dot - 5).c_str());
    if (i < 0 || i >= m->cfg.n_blocks) return fail(m, COSK_ERR_ARG, "bad block index in %s", name);
    std::string f = s.substr(dot + 1);
    BlockW &b = m->blk[i];
    if (f == "mix") b.mix = v;
    else if (f == "gcn.w") b.gcn_w = v;
    else if (f == "gcn.b") b.gcn_b = v;
    else if (f == "tcn.w") b.tcn_w = v;
    else if (f == "res.w") b.res_w = v;
    else if (f == "tcn.b") b.tcn_b = v;
    else if (f == "att.w") b.att_w = v;
    else if (f == "att.b") b.att_b = v;
    else if (f == "sa.in_scale") b.sa_scale = v;
    else if (f == "sa.in_shift") b.sa_shift = v;
    else if (f == "sa.qkv.w") b.sa_qkv_w = v;
    else if (f == "sa.qkv.b") b.sa_qkv_b = v;
    else if (f == "sa.skip_scale") b.sa_skip = v;
    else return fail(m, COSK_ERR_ARG, "unknown tensor %s", name);
  } else {
    return fail(m, COSK_ERR_ARG, "unknown tensor %s", name);
  }
  return COSK_OK;
}

int cosk_set_batch(cosk_model *m, int64_t n_streams) { return cosk_set_batch_ex(m, n_streams, 1); }

int cosk_set_batch_ex(cosk_model *m, int64_t n_streams, int32_t time_chunk) {
  if (!m) return COSK_ERR_ARG;
  Batch nb;
  int rc = batch_geometry(m, n_streams, time_chunk, nb);  // a refused call leaves the handle's batch as it was
  if (rc) return rc;
  DeviceGuard guard_(m->cfg.device);
  if (!m->prepared && (rc = prepare(m))) return rc;
  CK(cudaDeviceSynchronize());
  free_batch(m->batch);  // before the new one is allocated: the peak is the new state alone
  rc = alloc_batch(m, n_streams, time_chunk, nb);
  if (!rc) rc = zero_state(m, nb, 0);
  if (!rc && cudaDeviceSynchronize() != cudaSuccess) rc = fail(m, COSK_ERR_CUDA, "cosk_set_batch: zeroing the state failed");
  if (rc) {  // the handle stays without a batch until a cosk_set_batch succeeds
    free_batch(nb);
    return rc;
  }
  std::swap(m->batch, nb);
  return COSK_OK;
}

int cosk_reset(cosk_model *m) {
  if (!m) return COSK_ERR_ARG;
  if (m->batch.n_streams == 0) return fail(m, COSK_ERR_STATE, "cosk_reset before cosk_set_batch");
  DeviceGuard guard_(m->cfg.device);
  CK(cudaDeviceSynchronize());
  int rc = zero_state(m, m->batch, 0);
  if (rc) return rc;
  CK(cudaDeviceSynchronize());
  return COSK_OK;
}

// Shared entry checks of cosk_step / cosk_steps: call order, and the failure latch.  A step that stopped half way
// leaves the host counters ahead of the device state, and a fired pipeline watchdog (bounded mbarrier wait,
// ptx.cuh) makes every later result garbage: both refuse further steps until cosk_reset / cosk_set_batch.
static int step_entry(cosk_model *m, const char *what = "step") {
  if (m->batch.n_streams == 0) return fail(m, COSK_ERR_STATE, "%s before cosk_set_batch", what);
  if (!m->prepared) return fail(m, COSK_ERR_STATE, "weights changed after cosk_set_batch: call cosk_set_batch again");
  if (m->h_dbg && m->h_dbg[0] != 0) m->failed = true;  // written by the async copy behind an earlier emitting call
  if (m->failed) {
    if (m->h_dbg && m->h_dbg[0] != 0)
      return fail(m, COSK_ERR_STATE, "device pipeline watchdog fired (code 0x%08x): results since then are invalid; cosk_reset to continue",
                  m->h_dbg[0]);
    return fail(m, COSK_ERR_STATE, "an earlier step failed half way: state and schedule are out of step; cosk_reset to continue");
  }
  return COSK_OK;
}

int cosk_step(cosk_model *m, const float *x_dev, int64_t nc_stride, float *out_dev, int32_t *emitted, void *stream) {
  if (!m || !x_dev || !out_dev) return COSK_ERR_ARG;
  int rc = step_entry(m);
  if (rc) return rc;
  DeviceGuard guard_(m->cfg.device);
  int32_t cnt = 0;
  rc = walk(m, m->batch, x_dev, nc_stride, 0, 1, true, out_dev, 0, 1, &cnt, (cudaStream_t)stream);
  if ((rc = end_walks(m, rc, cnt, (cudaStream_t)stream))) return rc;
  if (emitted) *emitted = cnt;
  return COSK_OK;
}

int cosk_steps(cosk_model *m, const float *x_dev, int32_t T, float *out_dev, int64_t out_stride, int32_t max_out,
               int32_t *n_emitted, void *stream) {
  return cosk_steps_ex(m, x_dev, T, out_dev, out_stride, max_out, n_emitted, stream, 0);
}

int cosk_steps_ex(cosk_model *m, const float *x_dev, int32_t T, float *out_dev, int64_t out_stride, int32_t max_out,
                  int32_t *n_emitted, void *stream, int32_t pad_end) {
  if (!m || !x_dev || !out_dev || T < 0) return COSK_ERR_ARG;
  int rc = step_entry(m);
  if (rc) return rc;
  DeviceGuard guard_(m->cfg.device);
  const cudaStream_t s = (cudaStream_t)stream;
  Batch &bt = m->batch;
  int32_t cnt = 0;
  rc = walk_frames(m, bt, x_dev, (long long)T * m->cfg.vertices * m->cfg.persons, T, out_dev, out_stride, max_out, &cnt, s);
  if (pad_end) {
    // The clip is over: every temporal module flushes its end padding, module by module (first the blocks in order,
    // `padding` zero frames into each temporal conv, then `pool_padding` zero vectors into the pooling window).  What a
    // flush emits runs through the later stages at once (depth first), which yields the same output sequence as the
    // library's module-by-module order because every stage is a causal sequential machine.  Each flush is one frame and
    // walks frame by frame, whatever the time chunk.
    const int stages = m->cfg.n_blocks + 1;
    for (int st = 0; st < stages && !rc; ++st) {
      const int reps = st < m->cfg.n_blocks ? m->cfg.padding : (m->cfg.classes > 0 ? m->cfg.pool_padding : 0);
      for (int z = 0; z < reps && !rc; ++z) rc = walk(m, bt, nullptr, 0, 0, 1, true, out_dev, out_stride, max_out, &cnt, s, st);
    }
  }
  if ((rc = end_walks(m, rc, cnt, s))) return rc;
  // the padded frames are not part of the stream: the sequence ends here and the state starts over
  if (pad_end && (rc = zero_state(m, bt, s))) return rc;
  if (n_emitted) *n_emitted = cnt;
  return COSK_OK;
}

int64_t cosk_state_bytes(const cosk_model *m) { return m ? m->batch.state_bytes : 0; }

int cosk_last_schedule(const cosk_model *m, int32_t *flags, int32_t n) {
  if (!m || !flags || n < m->cfg.n_blocks + 1) return COSK_ERR_ARG;
  for (int i = 0; i <= m->cfg.n_blocks; ++i) flags[i] = m->batch.last_flags[i];
  return COSK_OK;
}

int64_t cosk_frame_count(const cosk_model *m) { return m ? m->batch.cnt.frame : 0; }

int cosk_read_block(cosk_model *m, int32_t block, float *dst_dev, void *stream) {
  if (!m || !dst_dev || block < 0 || block >= m->cfg.n_blocks) return COSK_ERR_ARG;
  const Batch &bt = m->batch;
  if (bt.n_streams == 0) return fail(m, COSK_ERR_STATE, "cosk_read_block before cosk_set_batch");
  const long long n_out = bt.cnt.n_out[block];
  if (n_out == 0) return fail(m, COSK_ERR_STATE, "block %d has not emitted yet", block);
  DeviceGuard guard_(m->cfg.device);
  return read_block(m, bt, bt.blk[block].out, (int)((n_out - 1) % bt.Ro), dst_dev, (cudaStream_t)stream);
}

int64_t cosk_launch_count(const cosk_model *m) { return m ? m->launches : 0; }

int cosk_block_uses_tensor_cores(const cosk_model *m, int32_t block) {
  if (!m || block < 0 || block >= m->cfg.n_blocks) return COSK_ERR_ARG;
  const Route &r = m->blk[block].route;
  return ((r.gcn_tc() || r.sa_out_tc) ? 1 : 0) | (r.tcn_tc ? 2 : 0);
}

int cosk_describe(const cosk_model *m, char *buf, size_t n) {
  if (!m || !buf || n < 2) return COSK_ERR_ARG;
  std::string o = "{";
  char t[1024];
  snprintf(t, sizeof t,
           "\"version\": \"%s\", \"path\": \"%s\", \"fuse_block\": %d, \"gcn_transposed\": %d, \"agcn_transposed\": %d, \"trace\": %d, ",
           cosk_version(), m->cfg.path == COSK_PATH_AUTO ? "auto" : "simt", m->fuse_block, m->gcn_transposed, m->agcn_transposed,
           m->d_trace ? 1 : 0);
  o += t;
  o += "\"blocks\": [";
  for (int i = 0; i < m->cfg.n_blocks; ++i) {
    const cosk_block_cfg &bc = m->cfg.blocks[i];
    const Route &r = m->blk[i].route;
    if (r.block64) {
      snprintf(t, sizeof t, "%s{\"block\": \"k_tc_block64 (graph conv + temporal conv in one kernel)\"}", i ? ", " : "");
      o += t;
      continue;
    }
    if (r.tcn_tc) snprintf(t, sizeof t, "%s<%d>", tcn_on_pair(m->batch, bc.cout) ? "k_tc_tcn2" : "k_tc_tcn", bc.cout);
    const std::string tc = r.tcn_tc ? t : "k_tcn_simt";
    snprintf(t, sizeof t, "%s{\"gcn\": \"%s\", \"tcn\": \"%s\"}", i ? ", " : "", gcn_name(m->blk[i]).c_str(), tc.c_str());
    o += t;
  }
  o += "], \"graph_conv\": {";
  bool firstw = true;
  for (int w : {64, 128, 256})
    for (int i = 0; i < m->cfg.n_blocks; ++i)
      if (m->cfg.blocks[i].cout == w && m->cfg.blocks[i].cin >= 64 && m->cfg.blocks[i].gconv == COSK_GCONV_PLAIN) {
        const GcnRoute g = m->blk[i].route.gcn;
        snprintf(t, sizeof t, "%s\"%d\": \"%s\"", firstw ? "" : ", ", w, g == GcnRoute::kTcT ? "gcnt" : g == GcnRoute::kTc ? "gcn" : "simt");
        o += t;
        firstw = false;
        break;
      }
  o += "}}";
  if (o.size() + 1 > n) return COSK_ERR_ARG;
  memcpy(buf, o.c_str(), o.size() + 1);
  return COSK_OK;
}

int cosk_device_error(cosk_model *m, uint32_t *code) {
  if (!m || !code) return COSK_ERR_ARG;
  DeviceGuard guard_(m->cfg.device);
  unsigned int h[4] = {0, 0, 0, 0};
  CK(cudaMemcpy(h, m->d_dbg, sizeof h, cudaMemcpyDeviceToHost));
  *code = h[0];
  return COSK_OK;
}

int cosk_simulate_schedule(const cosk_config *cfg, int32_t T, int32_t *flags) {
  if (!cfg || !flags || T < 0 || cfg->n_blocks < 1 || cfg->n_blocks > COSK_MAX_BLOCKS) return COSK_ERR_ARG;
  Counters k;
  for (int t = 0; t < T; ++t) schedule_frame(*cfg, k, flags + (size_t)t * (cfg->n_blocks + 1));
  return COSK_OK;
}

int cosk_schedule_compatible(const cosk_config *cfg, int64_t frame_a, int64_t frame_b) {
  if (!cfg || cfg->n_blocks < 1 || cfg->n_blocks > COSK_MAX_BLOCKS || frame_a < 0 || frame_b < 0) return COSK_ERR_ARG;
  if (cfg->padding < 0 || cfg->padding > kTaps - 1 || (cfg->classes > 0 && cfg->pool_size < 1)) return COSK_ERR_ARG;
  long long period = 1;
  for (int i = 0; i < cfg->n_blocks; ++i) {
    if (cfg->blocks[i].stride < 1) return COSK_ERR_ARG;
    period *= cfg->blocks[i].stride;
  }
  if (frame_a == frame_b) return 1;
  Counters a = counters_at(*cfg, frame_a), b = counters_at(*cfg, frame_b);
  // Compare the flags frame by frame until both counters are past the warm-up; from there on both schedules repeat with
  // the period (the product of the strides), so one more period decides every later frame.
  int32_t fa[COSK_MAX_BLOCKS + 1], fb[COSK_MAX_BLOCKS + 1];
  long long left = -1;
  while (left != 0) {
    schedule_frame(*cfg, a, fa);
    schedule_frame(*cfg, b, fb);
    if (memcmp(fa, fb, sizeof(int32_t) * (cfg->n_blocks + 1)) != 0) return 0;
    if (left > 0) --left;
    else if (past_warmup(*cfg, a) && past_warmup(*cfg, b)) left = period;
  }
  return 1;
}

int cosk_trace_read(cosk_model *m, uint64_t *out, int32_t n) {
  if (!m || !out || n < 1) return COSK_ERR_ARG;
  if (!m->d_trace) return fail(m, COSK_ERR_STATE, "tracing is off (set COSK_TRACE=1 before cosk_create)");
  DeviceGuard guard_(m->cfg.device);
  CK(cudaMemcpy(out, m->d_trace, sizeof(uint64_t) * (size_t)(n < 64 ? n : 64), cudaMemcpyDeviceToHost));
  return COSK_OK;
}

int cosk_profile_enable(cosk_model *m, int32_t on) {
  if (!m) return COSK_ERR_ARG;
  m->prof_on = on != 0;
  m->prof.clear();
  m->ev_used = 0;
  return COSK_OK;
}

int cosk_profile_read(cosk_model *m, int32_t kind, int32_t block, double *ms, int64_t *launches) {
  if (!m || !ms || !launches) return COSK_ERR_ARG;
  DeviceGuard guard_(m->cfg.device);
  double tot = 0.0;
  int64_t cnt = 0;
  for (size_t i = 0; i + 1 < m->prof.size(); ++i) {
    const ProfRec &r = m->prof[i];
    if (r.kind != kind || (block >= 0 && r.block != block)) continue;
    CK(cudaEventSynchronize(m->prof[i + 1].ev));
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, r.ev, m->prof[i + 1].ev));
    tot += t;
    ++cnt;
  }
  *ms = tot;
  *launches = cnt;
  return COSK_OK;
}

int64_t cosk_stream_bytes(const cosk_model *m) { return m ? state_args(m, m->batch).stream_bytes : 0; }

int cosk_reset_streams(cosk_model *m, const int64_t *idx, int64_t n, void *stream) {
  if (!m) return COSK_ERR_ARG;
  int rc = step_entry(m, "cosk_reset_streams");
  if (rc || (rc = check_indices(m, idx, n, 0, m->batch.n_streams, true))) return rc;
  DeviceGuard guard_(m->cfg.device);
  return launch_stream_state(m, m->batch, kStateZero, nullptr, (cudaStream_t)stream);
}

int cosk_export_streams(cosk_model *m, const int64_t *idx, int64_t n, void *dst_dev, cosk_stream_meta *meta, void *stream) {
  if (!m || !meta || (n > 0 && !dst_dev)) return COSK_ERR_ARG;
  int rc = step_entry(m, "cosk_export_streams");
  if (rc || (rc = check_indices(m, idx, n, 0, m->batch.n_streams, true))) return rc;
  DeviceGuard guard_(m->cfg.device);
  meta->abi_version = COSK_ABI_VERSION;
  meta->geometry = geometry_of(m->cfg);
  meta->frame = m->batch.cnt.frame;
  return launch_stream_state(m, m->batch, kStateGather, dst_dev, (cudaStream_t)stream);
}

int cosk_import_streams(cosk_model *m, const int64_t *idx, int64_t n, const void *src_dev, const cosk_stream_meta *meta,
                        void *stream) {
  if (!m || !meta || (n > 0 && !src_dev)) return COSK_ERR_ARG;
  int rc = step_entry(m, "cosk_import_streams");
  if (rc || (rc = check_indices(m, idx, n, 0, m->batch.n_streams, true))) return rc;
  if (meta->abi_version != COSK_ABI_VERSION || meta->geometry != geometry_of(m->cfg))
    return fail(m, COSK_ERR_STATE, "stream payload of another model geometry or library version");
  if (cosk_schedule_compatible(&m->cfg, meta->frame, m->batch.cnt.frame) != 1)
    return fail(m, COSK_ERR_STATE, "stream payload exported at frame %lld does not fit the schedule at frame %lld",
                (long long)meta->frame, m->batch.cnt.frame);
  DeviceGuard guard_(m->cfg.device);
  return launch_stream_state(m, m->batch, kStateScatter, const_cast<void *>(src_dev), (cudaStream_t)stream);
}

int cosk_resize_batch(cosk_model *m, int64_t n_streams, const int64_t *src) {
  if (!m) return COSK_ERR_ARG;
  int rc = step_entry(m, "cosk_resize_batch");
  if (rc) return rc;
  if (n_streams < 1 || !src) return fail(m, COSK_ERR_ARG, "cosk_resize_batch: n_streams %lld", (long long)n_streams);
  if ((rc = check_indices(m, src, n_streams, -1, m->batch.n_streams, false))) return rc;
  DeviceGuard guard_(m->cfg.device);
  CK(cudaDeviceSynchronize());  // no step or state call is in flight on the old buffers
  // The new batch keeps the time chunk, the counters and the last step's flags; it is filled from the old one and
  // installed only once that has worked.
  Batch nb;
  rc = alloc_batch(m, n_streams, m->batch.tchunk, nb);
  if (!rc) {
    nb.cnt = m->batch.cnt;
    memcpy(nb.last_flags, m->batch.last_flags, sizeof nb.last_flags);
    rc = zero_buffers(m, nb, 0);
  }
  if (!rc) rc = launch_stream_state(m, nb, kStateMove, nullptr, 0, &m->batch);
  if (!rc && cudaDeviceSynchronize() != cudaSuccess) rc = fail(m, COSK_ERR_CUDA, "cosk_resize_batch: state move failed");
  if (rc) cudaGetLastError();
  else std::swap(m->batch, nb);
  free_batch(nb);  // whichever batch lost
  return rc;
}

int cosk_prime_streams(cosk_model *m, const int64_t *idx, int64_t n, const float *x_dev, int32_t T, int32_t time_chunk,
                       void *stream) {
  if (!m) return COSK_ERR_ARG;
  Batch &bt = m->batch;
  int rc = step_entry(m, "cosk_prime_streams");
  if (rc || (rc = check_indices(m, idx, n, 0, bt.n_streams, true))) return rc;
  if (T < 0 || (n > 0 && T > 0 && !x_dev) || time_chunk < 1 || time_chunk > 4096)
    return fail(m, COSK_ERR_ARG, "cosk_prime_streams: T %d, time_chunk %d", (int)T, (int)time_chunk);
  if (n == 0) return COSK_OK;
  DeviceGuard guard_(m->cfg.device);
  const cudaStream_t s = (cudaStream_t)stream;
  const int H = (int)std::min<long long>(T, bt.cnt.frame);  // the handle's streams have not seen further back either
  if (H == 0) {
    if ((rc = launch_stream_state(m, bt, kStateZero, nullptr, s))) return rc;
    CK(cudaDeviceSynchronize());
    return COSK_OK;
  }
  const cosk_config &c = m->cfg;
  const std::vector<long long> dst = m->h_idx;
  const long long stream_bytes = state_args(m, bt).stream_bytes;
  const size_t out_elems = c.classes > 0 ? (size_t)n * c.classes : (size_t)n * c.persons * c.vertices * c.blocks[c.n_blocks - 1].cout;
  void *payload = nullptr;
  float *out = nullptr;
  uint32_t watchdog = 0;
  // The n streams walk on a scratch batch of their own, rings sized for `time_chunk`, from the counters of frame F - H.
  // The handle's batch is not touched before the scatter, so its time chunk, counters and flags stay as they were.
  Batch sb;
  rc = alloc_batch(m, n, time_chunk, sb);
  if (!rc) rc = zero_buffers(m, sb, s);
  if (!rc && (cudaMalloc(&payload, (size_t)n * stream_bytes) != cudaSuccess || cudaMalloc(&out, out_elems * sizeof(float)) != cudaSuccess))
    rc = fail(m, COSK_ERR_CUDA, "cosk_prime_streams: out of device memory for %lld streams", (long long)n);
  if (!rc) {
    sb.cnt = counters_at(c, bt.cnt.frame - H);
    int32_t cnt = 0;  // emissions all land in the one scratch output row
    rc = walk_frames(m, sb, x_dev + (long long)(T - H) * c.vertices * c.persons, (long long)T * c.vertices * c.persons, H, out, 0,
                     1, &cnt, s);
  }
  // The counters are a function of the frame count alone, so the walk ends where the handle stands and the scratch
  // streams' state fits the handle's schedule.  (Counters is all long long: no padding bytes to compare.)
  if (!rc && memcmp(&sb.cnt, &bt.cnt, sizeof sb.cnt) != 0)
    rc = fail(m, COSK_ERR_STATE, "cosk_prime_streams: walk ended off the handle's counters");
  if (!rc) {
    m->h_idx.resize((size_t)n);
    for (int64_t q = 0; q < n; ++q) m->h_idx[(size_t)q] = q;
    rc = launch_stream_state(m, sb, kStateGather, payload, s);
  }
  if (!rc && cudaMemcpyAsync(m->h_dbg, m->d_dbg, sizeof(unsigned int), cudaMemcpyDeviceToHost, s) != cudaSuccess)
    rc = fail(m, COSK_ERR_CUDA, "cudaMemcpyAsync of the watchdog word failed");
  if (!rc && cudaDeviceSynchronize() != cudaSuccess) rc = fail(m, COSK_ERR_CUDA, "cosk_prime_streams: priming walk failed");
  if (!rc) watchdog = m->h_dbg[0];
  if (rc) cudaGetLastError();
  free_batch(sb);
  if (!rc && watchdog) {
    m->failed = true;  // as after any walk: step_entry reports the code
    rc = fail(m, COSK_ERR_STATE, "device pipeline watchdog fired (code 0x%08x) while priming streams; cosk_reset to continue", watchdog);
  }
  if (!rc) {
    m->h_idx = dst;
    rc = launch_stream_state(m, bt, kStateScatter, payload, s);
  }
  if (!rc && cudaDeviceSynchronize() != cudaSuccess) rc = fail(m, COSK_ERR_CUDA, "cosk_prime_streams: scatter failed");
  dfree(payload);
  dfree(out);
  return rc;
}

}  // extern "C"
