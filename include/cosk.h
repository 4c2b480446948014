/*
 * cosk.h -- C ABI of libcosk: continual ST-GCN per-step forward on NVIDIA B200 (sm_100a).
 *
 * The reference (LukasHedegaard/continual-skeletons) has no FFI: its boundary for this path is the
 * Python `co.Module` protocol as used by `CoModelBase` (models/base.py:19-227).  Each entry point
 * below states the reference call it stands behind.  The library owns every weight and every
 * per-stream state buffer (temporal rings, delayed-residual rings, pooling window) on the device;
 * the caller owns input / output device buffers and passes raw pointers plus a CUDA stream.
 *
 * Conventions: every function returns 0 on success or a negative cosk_status; nothing throws
 * across the ABI; a handle is used from one host thread at a time (the reference mutates module
 * state in forward_step without locking); one handle per GPU.  There is no CPU fallback: without a
 * CUDA device cosk_create fails with COSK_ERR_CUDA.
 */
#ifndef COSK_H_
#define COSK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COSK_MAX_BLOCKS 16
#define COSK_ABI_VERSION 3

typedef struct cosk_model cosk_model;

enum cosk_status {
  COSK_OK = 0,
  COSK_ERR_ARG = -1,      /* bad argument / unsupported geometry */
  COSK_ERR_CUDA = -2,     /* CUDA runtime or driver error (see cosk_last_error) */
  COSK_ERR_STATE = -3,    /* call order (e.g. step before set_batch / missing weights) */
  COSK_ERR_UNSUPPORTED = -4
};

/* residual wiring of one CoSpatioTemporalBlock (models/base.py:412-446) */
enum cosk_res_kind { COSK_RES_NONE = 0, COSK_RES_IDENTITY = 1, COSK_RES_CONV = 2 };

/* kernel selection */
enum cosk_path {
  COSK_PATH_AUTO = 0, /* tcgen05 tile kernels wherever channels are multiples of 64, else SIMT */
  COSK_PATH_SIMT = 1  /* fp32 CUDA-core kernels everywhere: on-device checker, not the product */
};

/* graph convolution of a block */
enum cosk_graph_conv {
  COSK_GCONV_PLAIN = 0,    /* GraphConvolution: fixed sparse A * graph_attn (models/base.py:230-270) */
  COSK_GCONV_ADAPTIVE = 1, /* AdaptiveGraphConvolution: dense A + graph_attn plus a per-frame softmax vertex attention
                              (models/a_gcn/a_gcn.py:12-69, stepped by models/coa_gcn/coa_gcn.py:11-14) */
  COSK_GCONV_ATTENTION = 2 /* GcnUnitAttention, only_attention: 8-head self-attention over the V vertices of a frame
                              (models/s_tr/s_tr.py:19-231,303-476; layers 4-10 of models/cos_tr/cos_tr.py:24-41) */
};

typedef struct {
  int32_t cin, cout;
  int32_t stride;   /* temporal stride of tcn and residual conv: 1 or 2 */
  int32_t res_kind; /* enum cosk_res_kind */
  int32_t gconv;    /* enum cosk_graph_conv */
} cosk_block_cfg;

/* Geometry of a stack.  Mirrors what CoStGcn.__init__ / CoStGcnMod.__init__
 * (models/cost_gcn/cost_gcn.py:21-41, models/cost_gcn_mod/cost_gcn_mod.py:21-40) and
 * CoModelBase.on_init_end (models/base.py:68-122) fix at construction. */
typedef struct {
  int32_t abi_version;  /* COSK_ABI_VERSION */
  int32_t vertices;     /* V: 25 NTU, 18 Kinetics (datasets/datasets.py:128-134) */
  int32_t persons;      /* S / M: skeletons per stream, 2 */
  int32_t c_in;         /* input channels, 3 */
  int32_t n_blocks;
  int32_t padding;      /* temporal padding of every 9-tap conv: 4 ("equal") or 0 */
  int32_t classes;      /* 0: no head -- the last block's output is returned instead of logits */
  int32_t pool_size;    /* co.AvgPool1d window (models/base.py:86-97); ignored without head */
  int32_t pool_padding;
  int32_t data_bn;      /* 1: per-feature affine of data_bn (models/base.py:76) on the input */
  int32_t device;       /* CUDA device ordinal */
  int32_t path;         /* enum cosk_path */
  cosk_block_cfg blocks[COSK_MAX_BLOCKS];
} cosk_config;

/* Stands behind Model(hparams) construction.  Allocates weights (not state). */
int cosk_create(const cosk_config *cfg, cosk_model **out);
void cosk_destroy(cosk_model *m);

/* Stands behind load_state_dict (models/base.py:200-227 mapping is done by the host side, which
 * also folds eval-mode BatchNorm into the preceding conv).  `name` is one of
 *   "data_bn.scale" "data_bn.shift"            [S*V*C]   feature f = s*V*C + v*C + c
 *   "block<i>.mix"                             [3][V][V] A * graph_attn (models/base.py:262);
 *                                              A + graph_attn for COSK_GCONV_ADAPTIVE (models/a_gcn/a_gcn.py:50)
 *   "block<i>.att.w"  "block<i>.att.b"         [6*(cout/4)][cin], [6*(cout/4)]   COSK_GCONV_ADAPTIVE only: the embedding
 *                                              convs, rows theta_0, phi_0, theta_1, phi_1, theta_2, phi_2 (a_gcn.py:53-60)
 *   COSK_GCONV_ATTENTION blocks take, instead of mix / gcn.w as above:
 *   "block<i>.sa.in_scale" "block<i>.sa.in_shift"  [cin*V]  the unit's data_bn, feature c*V + v (s_tr.py:424-427)
 *   "block<i>.sa.qkv.w"  "block<i>.sa.qkv.b"   [2*dk + dv][cin], [2*dk + dv]  dk = cout/4, dv = cout, rows q | k | v with the
 *                                              dkh^-0.5 query scale folded in (s_tr.py:233-252)
 *   "block<i>.gcn.w"  "block<i>.gcn.b"         [cout][cout], [cout]  the output conv (s_tr.py:229-230) with the unit's bn folded
 *   "block<i>.sa.skip_scale"                   [cout]  scale of that bn: the skip connection x (cin == cout) is added before
 *                                              the bn (s_tr.py:464-470), i.e. enters as skip_scale[c] * x[c]
 *   "block<i>.gcn.w"                           [cout][3*cin (+cin if cin != cout)]  partition-major K
 *   "block<i>.gcn.b"                           [cout]
 *   "block<i>.tcn.w"                           [cout][9*cout]  tap-major K (tap 8 = newest frame)
 *   "block<i>.res.w"                           [cout][cin]     only res_kind == COSK_RES_CONV
 *   "block<i>.tcn.b"                           [cout]          tcn + residual-conv bias
 *   "fc.w" [classes][c_last]   "fc.b" [classes]
 * `host` is fp32 host memory that stays owned by the caller; n is the element count. */
int cosk_load_weights(cosk_model *m, const char *name, const float *host, size_t n);

/* Stands behind clean_state_on_shape_change (models/base.py:161-164): (re)allocates all state for
 * `n_streams` concurrent streams and zeroes it.  A refused call (COSK_ERR_ARG: a stream count or time chunk out of
 * range, or rings past 32-bit rows) leaves the handle as it was.  The old state is freed before the new state is
 * allocated; if allocating or zeroing it fails the handle has no batch, and every call that needs one returns
 * COSK_ERR_STATE until a cosk_set_batch succeeds. */
int cosk_set_batch(cosk_model *m, int64_t n_streams);
/* The same with a time chunk: cosk_steps then runs the stack module by module over chunks of up to `time_chunk` frames -- one
 * launch per kernel and chunk, its work items (frame, tile) pairs -- the way the library's forward_steps walks a clip
 * (models/base.py:187-190; SURVEY.md section 3.4).  The temporal rings hold 8 + time_chunk slots and the input / block-output
 * rings 4 + time_chunk (9 and 5 for time_chunk = 1, which is cosk_set_batch), so state grows with the chunk.  cosk_step is
 * unaffected.  Stacks with a kernel outside the tensor-core CoST-GCN path (SIMT blocks, adaptive / attention graph convs)
 * accept the call and step frame by frame. */
int cosk_set_batch_ex(cosk_model *m, int64_t n_streams, int32_t time_chunk);
/* Stands behind clean_state() (models/base.py:150,175): zero rings, delay lines, pool window and
 * every step counter. */
int cosk_reset(cosk_model *m);

/* Stands behind CoModelBase.forward_step (models/base.py:183-185).
 * x_dev: fp32 device pointer to one frame of all streams, logical shape (N, C, V, S); element
 *        (n, c, v, s) is read at x_dev[(n*C + c)*nc_stride + v*S + s]  (nc_stride = V*S for a
 *        contiguous frame, T*V*S for frame t of a (N,C,T,V,S) clip passed as x_dev + t*V*S).
 * out_dev: fp32 (N, classes) -- or (N*S, c_last, V) without head -- written iff *emitted == 1.
 * Asynchronous on `stream` (a cudaStream_t passed as void*); no host synchronisation. */
int cosk_step(cosk_model *m, const float *x_dev, int64_t nc_stride, float *out_dev, int32_t *emitted,
              void *stream);

/* Stands behind CoModelBase.forward_steps(pad_end=False) (models/base.py:187-190).
 * x_dev: (N, C, T, V, S) contiguous.  Emission e is written at out_dev + e*out_stride.
 * max_out bounds the number of emissions stored (later ones are computed but not stored). */
int cosk_steps(cosk_model *m, const float *x_dev, int32_t T, float *out_dev, int64_t out_stride,
               int32_t max_out, int32_t *n_emitted, void *stream);

/* forward_steps(pad_end=True) of the un-vendored continual-inference library, which the reference's own block tests use
 * (tests/test_cost_gcn.py:67,223,270,325): after the T frames every temporal module is fed its end padding -- `padding`
 * zero frames into each block's temporal conv, `pool_padding` zero vectors into the pooling window -- so that the emissions
 * equal the outputs of the regular zero-padded network on the whole clip.  The padded frames are not part of the stream:
 * the state is reset (as by cosk_reset, asynchronously on `stream`) when the call returns.  pad_end = 0: cosk_steps. */
int cosk_steps_ex(cosk_model *m, const float *x_dev, int32_t T, float *out_dev, int64_t out_stride,
                  int32_t max_out, int32_t *n_emitted, void *stream, int32_t pad_end);

/* Introspection (parity of the integer schedule, roofline accounting). */
int64_t cosk_state_bytes(const cosk_model *m);
/* flags[i] = 1 iff block i emitted during the last cosk_step; flags[n_blocks] = head emitted. */
int cosk_last_schedule(const cosk_model *m, int32_t *flags, int32_t n);
/* Host-only: the emission schedule of T consecutive frames from a fresh state, without touching a device
 * (same integer bookkeeping cosk_step uses).  flags is [T][n_blocks + 1], laid out like cosk_last_schedule. */
int cosk_simulate_schedule(const cosk_config *cfg, int32_t T, int32_t *flags);
/* Host-only: 1 iff the emission bookkeeping started from frame count frame_a and from frame_b gives identical flags on
 * every later frame, else 0 (negative: bad argument).  In practice: the counts are equal, or both are past the warm-up
 * after which the schedule repeats and they are congruent modulo the product of the block strides (the model's stride:
 * 4 for CoST-GCN, 1 for CoST-GCN*).  cosk_import_streams accepts a payload only between compatible frame counts. */
int cosk_schedule_compatible(const cosk_config *cfg, int64_t frame_a, int64_t frame_b);
/* frames pushed since the last reset */
int64_t cosk_frame_count(const cosk_model *m);

/* ---- per-stream state: a serving extension without counterpart in the reference ----------------------------------
 * All streams of a handle share one frame counter and one emission schedule; these calls act on the state of chosen
 * streams and never on the counters.  Index arrays are host memory of n int64 stream indices, checked on the host: an
 * index out of range, or an index that repeats within one call, returns COSK_ERR_ARG and launches nothing.  n = 0 is a
 * no-op.  Reset, export and import are one kernel launch each, asynchronous on `stream`, and never synchronise the host;
 * the indices reach the device through a handle-owned buffer.  Every call returns COSK_ERR_STATE before cosk_set_batch
 * and on a handle that has latched a failure (see cosk_step).
 *
 * Payload of one stream (cosk_stream_bytes bytes; rows of n streams are stored back to back).  Rings are stored in age
 * order, newest entry first, and hold only the entries a later step can read, so the payload is the same for every
 * time_chunk, stream count and tile position:
 *   input ring        4 entries (the delayed residual x_{n-4} of block 0) if block 0 has a residual, else none
 *   per block i:
 *     temporal ring   the 8 history taps of its 9-tap conv
 *     output ring     4 entries if block i+1 has a residual (its x_{n-4}), else 1 (the newest, cosk_read_block's rows)
 *   pooling window    with a head: pool_size entries of [c_last] fp32, then the fp64 running window sum [c_last]
 * A bf16 ring entry is its hi plane, then its lo plane, each [S*V tokens][round_up(c, 8)] bf16 (token s*V + v).  The
 * values are the raw planes, so export followed by import is bit-exact. */
typedef struct {
  int32_t abi_version; /* COSK_ABI_VERSION of the exporting library */
  uint64_t geometry;   /* fingerprint of every cosk_config field that shapes the payload or the meaning of its entries */
  int64_t frame;       /* the exporter's cosk_frame_count */
} cosk_stream_meta;
/* payload bytes per stream (valid before cosk_set_batch) */
int64_t cosk_stream_bytes(const cosk_model *m);
/* The listed streams' state becomes what cosk_reset leaves: zero rings and pooling window.  The counters stay, so the
 * streams predict on the handle's schedule at once, from zero history. */
int cosk_reset_streams(cosk_model *m, const int64_t *idx, int64_t n, void *stream);
/* Payload row q of dst_dev (device memory, n * cosk_stream_bytes bytes) := state of stream idx[q]; *meta describes it. */
int cosk_export_streams(cosk_model *m, const int64_t *idx, int64_t n, void *dst_dev, cosk_stream_meta *meta, void *stream);
/* State of stream idx[q] := payload row q of src_dev (device memory of this handle's device).  Refused with COSK_ERR_STATE,
 * the handle untouched, when meta's abi_version or geometry differ from this handle's, or when
 * cosk_schedule_compatible(cfg, meta->frame, cosk_frame_count) is 0.  Weights are not checked: a payload moved between
 * handles with different weights continues with this handle's weights. */
int cosk_import_streams(cosk_model *m, const int64_t *idx, int64_t n, const void *src_dev, const cosk_stream_meta *meta,
                        void *stream);
/* Changes the stream count to n_streams without cosk_set_batch's reset: new stream j takes old stream src[j]'s state
 * (src[j] = -1: zero state, as cosk_reset_streams leaves it).  src is host memory of n_streams entries; sources may
 * repeat.  The counters and the time chunk stay.  The new buffers are allocated and filled before the old ones are
 * freed, so the peak device memory is the state of both stream counts (cosk_state_bytes before + after); if an
 * allocation fails the handle stays exactly as it was.  Synchronises the device. */
int cosk_resize_batch(cosk_model *m, int64_t n_streams, const int64_t *src);
/* Primes joining streams from their recent frames.  x_dev: (n, C, T, V, S) contiguous fp32 device memory, row q the
 * history of stream idx[q], frame T-1 the newest (the one the other streams received at cosk_frame_count - 1).  With
 * F = cosk_frame_count and H = min(T, F), stream idx[q] ends with exactly the state it would have if cosk_reset_streams
 * had been called at frame F - H and the stream had then received frames T-H .. T-1 of its row; the oldest T - H frames
 * are ignored (the handle's streams have not seen further back either), and T = 0 is cosk_reset_streams.  With
 * H >= the receptive field a primed stream equals a stream that received those frames in the handle all along.  The
 * frames are walked as cosk_steps walks a clip on a handle of n streams with time chunk `time_chunk` (1: as cosk_step
 * walks them), on scratch state of their own, which is then gathered into a payload and scattered into idx.  Every
 * other stream's state, the counters, cosk_last_schedule's flags and the time chunk stay as they were; the primed
 * streams emit on the handle's schedule.  Refused (COSK_ERR_ARG / COSK_ERR_STATE / COSK_ERR_CUDA) with the handle
 * untouched on the index checks above, before cosk_set_batch, on a latched handle and when an allocation fails; a
 * pipeline watchdog firing during the walk latches the handle as a step would.  Peak device memory: the handle's
 * state, plus the state of n streams at time_chunk (as cosk_set_batch_ex(n, time_chunk) allocates), plus
 * n * cosk_stream_bytes, plus one output row of n streams.  Synchronises the device. */
int cosk_prime_streams(cosk_model *m, const int64_t *idx, int64_t n, const float *x_dev, int32_t T, int32_t time_chunk,
                       void *stream);
/* last emitted output of block i as fp32 (N*S, cout, V) into dst_dev (debug / feature taps) */
int cosk_read_block(cosk_model *m, int32_t block, float *dst_dev, void *stream);
/* kernels launched by this handle since creation */
int64_t cosk_launch_count(const cosk_model *m);
/* 1 iff block i runs on the tcgen05 kernels (bit 0: graph conv -- for a COSK_GCONV_ATTENTION block the unit's output
 * conv; its qkv conv and the attention itself run on CUDA cores --, bit 1: temporal conv) */
int cosk_block_uses_tensor_cores(const cosk_model *m, int32_t block);

/* Per-kernel-kind device timing with CUDA events on the launching stream.
 * kinds: 0 input, 1 gcn, 2 tcn, 3 pool+fc, 4 attention half of the adaptive gcn, 5 fused block step (graph conv + temporal
 * conv of a 64 -> 64 block in one kernel); enable before the timed region, then read. */
int cosk_profile_enable(cosk_model *m, int32_t on);
/* Sums the event-measured device time (ms) and launch count of (kind, block) since enable;
 * block < 0 sums over blocks.  Synchronises the recorded events. */
int cosk_profile_read(cosk_model *m, int32_t kind, int32_t block, double *ms, int64_t *launches);

/* First pipeline-watchdog code a tcgen05 kernel recorded since the last reset (0 = none).  A
 * non-zero code means a bounded mbarrier wait expired: results are invalid.  Synchronises. */
int cosk_device_error(cosk_model *m, uint32_t *code);

/* Phase timers (SM clock cycles, CTA 0) of the last graph-conv launch when the handle was created with
 * COSK_TRACE=1 in the environment: [0..3] drain warp {wait accumulator, tmem load + fold, wait exchange
 * buffer, write planes}, [5] drain total, [6] work items, [8..9] mix warp {wait planes, gather + store},
 * [16..18] MMA thread {wait accumulator free, wait operands, total}.  Debug aid. */
int cosk_trace_read(cosk_model *m, uint64_t *out, int32_t n);

/* The kernel selection this handle runs with, as a JSON object in `buf` (NUL-terminated, at most n bytes): the value of
 * every runtime knob read from the COSK_* environment at cosk_create and, per block, which graph-conv / temporal-conv
 * kernel serves it.  Valid after cosk_set_batch (weights prepared).  bench.py echoes it in its JSON line, so the
 * configuration behind a measured number is on record. */
int cosk_describe(const cosk_model *m, char *buf, size_t n);

const char *cosk_last_error(const cosk_model *m);
const char *cosk_version(void);

#ifdef __cplusplus
}
#endif
#endif /* COSK_H_ */
