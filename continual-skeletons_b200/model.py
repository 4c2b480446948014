"""Host-side mirror of the reference's continual model interface for the CoST-GCN hot path.

``CoStGcn`` / ``CoStGcnMod`` present what ``CoModelBase`` presents in the reference
(models/base.py:19-227): ``Model(hparams)``, ``forward_step`` / ``forward_steps`` / ``forward``,
``clean_state``, ``state_dict`` / ``load_state_dict`` / ``map_state_dict`` with the same nested
parameter names (so non-continual ST-GCN checkpoints load through the same key mapping),
``input_shape`` / ``output_shape`` / ``receptive_field`` / ``stride`` / ``padding`` / ``delay`` /
``call_mode`` / ``layers.layer1..10``.  The torch modules held here are parameter containers only:
every step runs in ``libcosk.so`` (include/cosk.h), which owns all per-stream state on the GPU.
There is no CPU path.
"""
import ctypes
import math
from collections import OrderedDict, namedtuple

import numpy as np
import torch
import torch.nn as nn

from . import graph as _graph
from . import lib as _lib
from .lib import CoskError

BN_EPS = 1e-5
KT = 9


GCONV_KINDS = {"plain": 0, "adaptive": 1, "attention": 2}  # enum cosk_graph_conv


class BlockSpec(namedtuple("BlockSpec", "cin cout stride residual gconv")):
    """One CoSpatioTemporalBlock (models/base.py:390-446).  ``gconv``: which graph conv it holds -- "plain"
    (GraphConvolution), "adaptive" (AdaptiveGraphConvolution), "attention" (GcnUnitAttention); "" takes the
    stack's default."""

    def __new__(cls, cin, cout, stride=1, residual=True, gconv=""):
        return super().__new__(cls, int(cin), int(cout), int(stride), bool(residual), str(gconv))

    @property
    def res_kind(self):
        if not self.residual:
            return 0
        return 1 if (self.cin == self.cout and self.stride == 1) else 2


StreamMeta = namedtuple("StreamMeta", "abi_version geometry frame")
StreamMeta.__doc__ = """cosk_stream_meta: library ABI version, geometry fingerprint and frame count of an exported payload."""


class StreamState(namedtuple("StreamState", "payload meta")):
    """State of some streams taken by ``export_streams``: ``payload`` is a CUDA uint8 tensor (n, stream_bytes), row q the
    q-th exported stream in the layout include/cosk.h documents; ``meta`` a ``StreamMeta``."""


class AttributeDict(dict):
    __getattr__ = dict.__getitem__
    __setattr__ = dict.__setitem__


class Configs:
    """Minimal stand-in for ``ride.Configs``: the reference's tests build hparams with
    ``Model.configs().default_values()`` (tests/test_cost_gcn.py:18-23)."""

    def __init__(self):
        self._d = OrderedDict()

    def add(self, name, default=None, **_):
        self._d[name] = default

    @property
    def names(self):
        return list(self._d)

    def default_values(self):
        return dict(self._d)


# datasets/datasets.py:128-134: name -> (classes, graph factory)
DATASETS = {
    "ntu60": (60, _graph.ntu_graph),
    "ntu120": (120, _graph.ntu_graph),
    "kinetics": (400, _graph.kinetics_graph),
    "dummy_ntu": (60, _graph.ntu_graph),
    "dummy_kin": (400, _graph.kinetics_graph),
}


# ---------------------------------------------------------------------------------------------
# parameter containers with the reference's names and initialisation
# ---------------------------------------------------------------------------------------------
def _init_conv(conv, bs=1):
    """models/utils.py:10-19."""
    nn.init.constant_(conv.bias, 0)
    if bs == 1:
        nn.init.kaiming_normal_(conv.weight, mode="fan_out")
    else:
        nn.init.normal_(conv.weight, 0, math.sqrt(2.0 / (conv.weight.numel() * bs)))


def _init_bn(bn, scale):
    """models/utils.py:20-22."""
    nn.init.constant_(bn.weight, scale)
    nn.init.constant_(bn.bias, 0)


class _Node(nn.Module):
    """Anonymous container; children are attached with ``add_module`` under the reference's names."""


def _gcn_params(cin, cout, A):
    """Parameters of GraphConvolution (models/base.py:231-258)."""
    g = _Node()
    a = torch.from_numpy(np.asarray(A, dtype=np.float32))
    g.graph_attn = nn.Parameter(torch.ones_like(a))
    g.A = nn.Parameter(a.clone(), requires_grad=False)
    g.g_conv = nn.ModuleList(nn.Conv2d(cin, cout, 1) for _ in range(3))
    for conv in g.g_conv:
        _init_conv(conv, bs=3)
    if cin != cout:
        g.gcn_residual = nn.Sequential(nn.Conv2d(cin, cout, 1), nn.BatchNorm2d(cout))
        _init_conv(g.gcn_residual[0], 1)
        _init_bn(g.gcn_residual[1], 1)
    g.bn = nn.BatchNorm2d(cout)
    _init_bn(g.bn, 1e-6)
    return g


def _agcn_params(cin, cout, A, coff_embedding=4):
    """Parameters of AdaptiveGraphConvolution (models/a_gcn/a_gcn.py:13-46): the plain graph conv's tensors plus
    the two embedding convs per partition; ``graph_attn`` is an additive dense term initialised to 1."""
    g = _gcn_params(cin, cout, A)
    inter_c = cout // coff_embedding
    if inter_c < 1:
        raise ValueError("AdaptiveGraphConvolution needs out_channels >= 4")
    g.a_conv = nn.ModuleList(nn.Conv2d(cin, inter_c, 1) for _ in range(3))
    g.b_conv = nn.ModuleList(nn.Conv2d(cin, inter_c, 1) for _ in range(3))
    for conv in list(g.a_conv) + list(g.b_conv):
        _init_conv(conv, 1)
    g.inter_c = inter_c
    return g


def _sa_params(cin, cout, A, V, heads=8):
    """Parameters of GcnUnitAttention(only_attention=True) + its SpatialAttention (models/s_tr/s_tr.py:303-415,
    26-101): per-(channel, vertex) input BatchNorm, qkv and output 1x1 convs with PyTorch's default init (the
    reference never re-initialises them), output BatchNorm, and the (unused here) parameter A."""
    dk, dv = int(cout * 0.25), cout
    if dk % heads or dv % heads or dk == 0:
        raise ValueError("GcnUnitAttention needs out_channels to be a multiple of 32 (dk = out/4 over 8 heads)")
    g = _Node()
    g.data_bn = nn.BatchNorm1d(cin * V)
    g.bn = nn.BatchNorm2d(cout)
    g.A = nn.Parameter(torch.from_numpy(np.asarray(A, dtype=np.float32)).clone())
    att = _Node()
    att.qkv_conv = nn.Conv2d(cin, 2 * dk + dv, 1)
    att.attn_out = nn.Conv2d(dv, dv, 1)
    g.attention_conv = att
    g.heads, g.dk, g.dv = heads, dk, dv
    return g


def _tconv_params(cin, cout, k, stride, pad):
    """Parameters of (Co)TemporalConvolution (models/base.py:279-334)."""
    t = _Node()
    t.t_conv = nn.Conv2d(cin, cout, kernel_size=(k, 1), padding=(pad, 0), stride=(stride, 1))
    t.bn = nn.BatchNorm2d(cout)
    _init_conv(t.t_conv, 1)
    _init_bn(t.bn, 1)
    return t


def _block_params(spec, A, pad, gconv="plain"):
    """Module tree with the state_dict keys of CoSpatioTemporalBlock (models/base.py:412-446):
    plain ``gcn.* / tcn.*`` without residual, ``0.1.gcn.* / 0.1.tcn.*`` under a residual wrapper,
    plus ``0.0.residual.*`` for the strided 1x1 residual conv."""
    if gconv == "attention":
        gcn = _sa_params(spec.cin, spec.cout, A, np.asarray(A).shape[-1])
    else:
        gcn = (_agcn_params if gconv == "adaptive" else _gcn_params)(spec.cin, spec.cout, A)
    tcn = _tconv_params(spec.cout, spec.cout, KT, spec.stride, pad)
    blk = _Node()
    if spec.res_kind == 0:
        blk.gcn, blk.tcn = gcn, tcn
        blk._cosk_parts = (gcn, tcn, None)
        return blk
    outer, main = _Node(), _Node()
    main.gcn, main.tcn = gcn, tcn
    res = None
    if spec.res_kind == 2:
        branch = _Node()
        res = _tconv_params(spec.cin, spec.cout, 1, spec.stride, 0)
        branch.residual = res
        outer.add_module("0", branch)
    outer.add_module("1", main)
    blk.add_module("0", outer)
    blk._cosk_parts = (gcn, tcn, res)
    return blk


def _fold_bn(bn):
    s = bn.weight.detach().double() / torch.sqrt(bn.running_var.detach().double() + BN_EPS)
    return s, bn.bias.detach().double() - bn.running_mean.detach().double() * s


def _folded_block_tensors(blk, spec):
    """BN-folded fp32 tensors in the layout cosk_load_weights documents (include/cosk.h)."""
    gcn, tcn, res = blk._cosk_parts
    if hasattr(gcn, "attention_conv"):
        out = _folded_attention_unit(gcn)
        out.update(_folded_temporal(tcn, res, spec))
        return {k: v.float().contiguous().cpu() for k, v in out.items()}
    s, t = _fold_bn(gcn.bn)
    ws = [conv.weight.detach().double()[:, :, 0, 0] * s[:, None] for conv in gcn.g_conv]
    bias = s * sum(conv.bias.detach().double() for conv in gcn.g_conv) + t
    if spec.cin != spec.cout:
        sr, tr = _fold_bn(gcn.gcn_residual[1])
        ws.append(gcn.gcn_residual[0].weight.detach().double()[:, :, 0, 0] * sr[:, None])
        bias = bias + sr * gcn.gcn_residual[0].bias.detach().double() + tr
    adaptive = hasattr(gcn, "a_conv")
    out = {
        # models/base.py:262 masks A with graph_attn; models/a_gcn/a_gcn.py:50 adds it
        "mix": (gcn.A.detach().double() + gcn.graph_attn.detach().double()) if adaptive
        else (gcn.A.detach().double() * gcn.graph_attn.detach().double()),
        "gcn.w": torch.cat(ws, dim=1),
        "gcn.b": bias,
    }
    if adaptive:  # rows: theta_0, phi_0, theta_1, phi_1, theta_2, phi_2 (a_gcn.py:53-60)
        convs = [c for pair in zip(gcn.a_conv, gcn.b_conv) for c in pair]
        out["att.w"] = torch.cat([c.weight.detach().double()[:, :, 0, 0] for c in convs], dim=0)
        out["att.b"] = torch.cat([c.bias.detach().double() for c in convs], dim=0)
    out.update(_folded_temporal(tcn, res, spec))
    return {k: v.float().contiguous().cpu() for k, v in out.items()}


def _folded_temporal(tcn, res, spec):
    """Temporal conv + block residual conv with their BatchNorms folded (models/base.py:307-334, 412-446)."""
    out = {}
    s, t = _fold_bn(tcn.bn)
    w = tcn.t_conv.weight.detach().double()[:, :, :, 0].permute(0, 2, 1) * s[:, None, None]  # [cout][tap][cin]
    out["tcn.w"] = w.reshape(spec.cout, KT * spec.cout)
    bias = s * tcn.t_conv.bias.detach().double() + t
    if res is not None:
        sr, tr = _fold_bn(res.bn)
        out["res.w"] = res.t_conv.weight.detach().double()[:, :, 0, 0] * sr[:, None]
        bias = bias + sr * res.t_conv.bias.detach().double() + tr
    out["tcn.b"] = bias
    return out


def _folded_attention_unit(gcn):
    """Tensors of a COSK_GCONV_ATTENTION block (include/cosk.h): the unit's data_bn as a per-(channel, vertex) affine,
    the qkv conv with the query scale dkh^-0.5 folded into its q rows (models/s_tr/s_tr.py:251-252), and the output
    conv with the unit's bn folded."""
    s_in, t_in = _fold_bn(gcn.data_bn)
    att = gcn.attention_conv
    wq = att.qkv_conv.weight.detach().double()[:, :, 0, 0].clone()
    bq = att.qkv_conv.bias.detach().double().clone()
    scale = float(gcn.dk // gcn.heads) ** -0.5
    wq[: gcn.dk] *= scale
    bq[: gcn.dk] *= scale
    s, t = _fold_bn(gcn.bn)
    return {
        "sa.in_scale": s_in, "sa.in_shift": t_in,
        "sa.qkv.w": wq, "sa.qkv.b": bq,
        "gcn.w": att.attn_out.weight.detach().double()[:, :, 0, 0] * s[:, None],
        "gcn.b": s * att.attn_out.bias.detach().double() + t,
        # the skip connection is added BEFORE the unit's bn (s_tr.py:464-470), so it carries the bn scale
        "sa.skip_scale": s,
    }


# ---------------------------------------------------------------------------------------------
# engine: one libcosk handle + the geometry it was built for
# ---------------------------------------------------------------------------------------------
class _Engine:
    def __init__(self, owner, device):
        self.lib = _lib.load_library()
        if not torch.cuda.is_available():
            raise CoskError("continual_skeletons_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise CoskError(f"continual_skeletons_b200 runs on CUDA devices only, got {self.device}")
        cfg = owner._config()
        cfg.device = self.device.index if self.device.index is not None else torch.cuda.current_device()
        h = ctypes.c_void_p()
        rc = self.lib.cosk_create(ctypes.byref(cfg), ctypes.byref(h))
        if rc != 0:
            raise CoskError(f"cosk_create failed with status {rc} (needs an sm_100a GPU)")
        self.h = h
        self.n_streams = None
        self.n_blocks = len(owner._specs)

    def check(self, rc, what):
        if rc != 0:
            msg = self.lib.cosk_last_error(self.h)
            raise CoskError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    def load(self, name, tensor):
        t = tensor.detach().float().contiguous().cpu()
        self.check(self.lib.cosk_load_weights(self.h, name.encode(), ctypes.c_void_p(t.data_ptr()), t.numel()), name)

    def close(self):
        if getattr(self, "h", None):
            self.lib.cosk_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _CoBase(nn.Module):
    """Shared machinery of the full models and the headless block stack."""

    def _setup(self, specs, pad, V, S, c_in, classes, head, A, path, adaptive=False):
        default = "adaptive" if adaptive else "plain"
        specs = [sp if sp.gconv else sp._replace(gconv=default) for sp in specs]
        for sp in specs:
            if sp.gconv not in GCONV_KINDS:
                raise ValueError(f"unknown graph conv kind {sp.gconv!r}")
        self._specs, self._pad, self._V, self._S, self._c_in = list(specs), int(pad), int(V), int(S), int(c_in)
        self._classes, self._head, self._path = int(classes), bool(head), path
        self._engine, self._dirty, self._shape = None, True, None
        # co.Sequential algebra over the blocks (SURVEY.md section 3.3)
        rf, cum, p = 1, 1, 0
        for sp in self._specs:
            rf += (KT - 1) * cum
            p += self._pad * cum
            cum *= sp.stride
        self.receptive_field, self.stride, self.padding = rf, cum, p
        self.delay = rf - 1 - p

    def _config(self):
        """The cosk_config of this stack (include/cosk.h)."""
        cfg = _lib.Config()
        cfg.abi_version = _lib.ABI_VERSION
        cfg.vertices, cfg.persons, cfg.c_in = self._V, self._S, self._c_in
        cfg.n_blocks, cfg.padding = len(self._specs), self._pad
        cfg.classes = self._classes if self._head else 0
        cfg.pool_size, cfg.pool_padding = (self.pool_size, self.pool_padding) if self._head else (0, 0)
        cfg.data_bn = 1 if self._head else 0
        cfg.path = {"auto": 0, "simt": 1}[self._path]
        for i, sp in enumerate(self._specs):
            cfg.blocks[i].cin, cfg.blocks[i].cout = sp.cin, sp.cout
            cfg.blocks[i].stride, cfg.blocks[i].res_kind = sp.stride, sp.res_kind
            cfg.blocks[i].gconv = GCONV_KINDS[sp.gconv]
        return cfg

    def simulate_schedule(self, frames):
        """Emission flags (one per block + head) of ``frames`` consecutive steps from a fresh state, computed
        by the library's host-side bookkeeping without a GPU."""
        lib = _lib.load_library()
        cfg = self._config()
        w = len(self._specs) + 1
        buf = (ctypes.c_int32 * (frames * w))()
        rc = lib.cosk_simulate_schedule(ctypes.byref(cfg), frames, buf)
        if rc != 0:
            raise CoskError(f"cosk_simulate_schedule failed ({rc})")
        return [tuple(bool(buf[t * w + i]) for i in range(w)) for t in range(frames)]

    # -- weights ------------------------------------------------------------------------------
    def _block_modules(self):
        raise NotImplementedError

    def _sync(self, device):
        if self._engine is not None and self._engine.device != torch.device(device):
            self._engine.close()
            self._engine = None
        if self._engine is None:
            self._engine = _Engine(self, device)
            self._dirty = True
        if self._dirty:
            e = self._engine
            for i, (blk, sp) in enumerate(zip(self._block_modules(), self._specs)):
                for k, v in _folded_block_tensors(blk, sp).items():
                    e.load(f"block{i}.{k}", v)
            if self._head:
                s, t = _fold_bn(self.data_bn)
                e.load("data_bn.scale", s)
                e.load("data_bn.shift", t)
                e.load("fc.w", self.fc.weight)
                e.load("fc.b", self.fc.bias)
            self._dirty = False
            self._shape = None  # new weights -> state is re-created on the next step
        return self._engine

    def sync_weights(self):
        """Re-fold and re-upload the parameters (call after editing them in place)."""
        self._dirty = True

    def load_state_dict(self, state_dict, strict=True, **kw):
        r = super().load_state_dict(state_dict, strict=strict, **kw)
        self._dirty = True
        return r

    def _apply(self, fn, *a, **kw):
        r = super()._apply(fn, *a, **kw)
        self._dirty = True
        return r

    # -- state --------------------------------------------------------------------------------
    def clean_state(self):
        """Zero every ring, delay line, pooling window and counter (models/base.py:150,175)."""
        if self._engine is not None and self._engine.n_streams is not None:
            self._engine.check(self._engine.lib.cosk_reset(self._engine.h), "cosk_reset")

    # -- per-stream state (a serving extension: the reference only resets all streams at once) ---------------------
    def _stream_engine(self, what):
        e = self._engine
        if e is None or e.n_streams is None or self._shape is None:
            raise CoskError(f"{what}: the model holds no stream state yet (step it first)")
        return e

    @staticmethod
    def _index_array(indices):
        idx = np.ascontiguousarray(np.asarray(indices, dtype=np.int64).reshape(-1))
        return idx, idx.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))

    @staticmethod
    def _device_stream(e):
        return ctypes.c_void_p(torch.cuda.current_stream(e.device).cuda_stream)

    def schedule_compatible(self, frame_a, frame_b):
        """True iff the emission schedule continues identically from frame counts ``frame_a`` and ``frame_b``
        (cosk_schedule_compatible; host only): the frames between which ``import_streams`` accepts a payload."""
        rc = _lib.load_library().cosk_schedule_compatible(ctypes.byref(self._config()), int(frame_a), int(frame_b))
        if rc < 0:
            raise CoskError(f"cosk_schedule_compatible failed ({rc})")
        return rc == 1

    def frame_count(self):
        """Frames pushed since the state was last reset as a whole."""
        return int(self._engine.lib.cosk_frame_count(self._engine.h)) if self._engine else 0

    def stream_bytes(self):
        """Bytes of one stream's exported state."""
        e = self._sync(torch.device("cuda", torch.cuda.current_device()) if self._engine is None else self._engine.device)
        return int(e.lib.cosk_stream_bytes(e.h))

    def reset_streams(self, indices):
        """Zero the state of the listed streams, as ``clean_state`` would, leaving every other stream and the shared
        frame counter alone.  The streams predict on the shared schedule at once, from zero history."""
        e = self._stream_engine("reset_streams")
        idx, p = self._index_array(indices)
        e.check(e.lib.cosk_reset_streams(e.h, p, idx.size, self._device_stream(e)), "cosk_reset_streams")

    def export_streams(self, indices):
        """The state of the listed streams as a ``StreamState`` (one payload row per index, in order)."""
        e = self._stream_engine("export_streams")
        idx, p = self._index_array(indices)
        payload = torch.empty((idx.size, int(e.lib.cosk_stream_bytes(e.h))), dtype=torch.uint8, device=e.device)
        meta = _lib.StreamMeta()
        e.check(e.lib.cosk_export_streams(e.h, p, idx.size, ctypes.c_void_p(payload.data_ptr()), ctypes.byref(meta),
                                          self._device_stream(e)), "cosk_export_streams")
        return StreamState(payload, StreamMeta(int(meta.abi_version), int(meta.geometry), int(meta.frame)))

    def import_streams(self, indices, state):
        """Overwrite the state of the listed streams with the rows of ``state`` (from ``export_streams`` of a model with the
        same geometry at a compatible frame count, see ``schedule_compatible``; any device).  Raises ``CoskError`` and
        leaves the state untouched otherwise."""
        e = self._stream_engine("import_streams")
        idx, p = self._index_array(indices)
        payload = state.payload
        if payload.dtype != torch.uint8 or payload.dim() != 2 or payload.shape[0] != idx.size or \
                payload.shape[1] != int(e.lib.cosk_stream_bytes(e.h)):
            raise CoskError(f"import_streams: payload of shape {tuple(payload.shape)} for {idx.size} streams")
        payload = payload.to(e.device).contiguous()
        meta = _lib.StreamMeta(*state.meta)
        e.check(e.lib.cosk_import_streams(e.h, p, idx.size, ctypes.c_void_p(payload.data_ptr()), ctypes.byref(meta),
                                          self._device_stream(e)), "cosk_import_streams")

    def resize_streams(self, keep):
        """Change the number of streams to ``len(keep)`` without a reset: new stream j continues old stream ``keep[j]``,
        or starts from zero state where ``keep[j]`` is -1.  The next ``forward_step`` / ``forward_steps`` with
        ``len(keep)`` streams continues on the shared schedule.  Peak device memory: the state of both stream counts."""
        e = self._stream_engine("resize_streams")
        idx, p = self._index_array(keep)
        e.check(e.lib.cosk_resize_batch(e.h, idx.size, p), "cosk_resize_batch")
        e.n_streams = int(idx.size)
        self._shape = (int(idx.size),) + tuple(self._shape[1:])

    def prime_streams(self, indices, clip):
        """Give the listed streams the state their recent frames leave.  ``clip``: (k, C, H, V, S) -- (k, C, H, V) for
        ``CoStack`` -- on the model's device, row j the history of stream ``indices[j]``, frame H - 1 the newest (the
        frame the other streams received last).  With F = ``frame_count()`` and H' = min(H, F), each stream ends as if
        ``reset_streams`` had been called at frame F - H' and it had then received the last H' frames of its row; older
        frames are ignored.  With H' >= ``receptive_field`` the stream equals one that received those frames here all
        along.  Every other stream, the frame count and the schedule stay as they were.  The frames are walked in chunks
        of ``_pick_time_chunk(k, H)``.  Synchronises the device; peak memory: the state of k streams at that chunk plus
        k * ``stream_bytes()`` on top of the model's own state."""
        e = self._stream_engine("prime_streams")
        idx, p = self._index_array(indices)
        want = (idx.size, self._shape[1], None) + tuple(self._shape[2:])
        if not isinstance(clip, torch.Tensor) or clip.dim() != len(want) or \
                any(w is not None and g != w for g, w in zip(clip.shape, want)):
            raise CoskError(f"prime_streams: clip of shape {tuple(getattr(clip, 'shape', ()))} for {idx.size} streams, "
                            f"expected {tuple('H' if w is None else w for w in want)}")
        if clip.device != e.device:
            raise CoskError(f"prime_streams: clip on {clip.device}, the model steps on {e.device}")
        x = self._check_input(clip, len(want))
        H = int(x.shape[2])
        e.check(e.lib.cosk_prime_streams(e.h, p, idx.size, ctypes.c_void_p(x.data_ptr()), H,
                                         self._pick_time_chunk(idx.size, H), self._stream(x)), "cosk_prime_streams")

    def _pick_time_chunk(self, n_streams, frames):
        """Frames per launch of forward_steps (cosk_set_batch_ex).  ``time_chunk`` > 0 is taken as given; auto (-1): the whole
        call in one chunk when the extra ring slots fit a budget (a quarter of the free device memory, at most 8 GiB), else
        as many frames as do; 1 when the state is first created by a single-frame call."""
        tc = int(getattr(self, "_time_chunk", -1))
        if tc > 0:
            return tc
        if frames <= 1:
            return 1
        per_frame = n_streams * self._S * self._V * 4 * 2 * sum(sp.cout for sp in self._specs)  # one more slot in every ring
        free, _ = torch.cuda.mem_get_info(self._engine.device)
        budget = min(8 << 30, free // 4)
        return int(max(1, min(frames, budget // max(per_frame, 1), 4096)))

    def _ensure_batch(self, e, shape, n_streams, frames=1):
        # models/base.py:161-164: any change of the per-step input shape resets all state
        if self._shape != shape or e.n_streams != n_streams:
            tc = self._pick_time_chunk(n_streams, frames)
            e.check(e.lib.cosk_set_batch_ex(e.h, int(n_streams), tc), "cosk_set_batch_ex")
            e.n_streams = int(n_streams)
            e.time_chunk = tc
            self._shape = shape

    @staticmethod
    def _check_input(x, ndim):
        if not isinstance(x, torch.Tensor) or x.dim() != ndim:
            raise ValueError(f"expected a {ndim}-d tensor, got {tuple(getattr(x, 'shape', ()))}")
        if x.device.type != "cuda":
            raise CoskError("inputs must live on the CUDA device that steps the model (no CPU path)")
        if x.dtype != torch.float32:
            x = x.float()
        return x.contiguous()

    def _stream(self, x):
        return ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)

    # -- introspection ------------------------------------------------------------------------
    def last_schedule(self):
        """Emit flags of the last step: one per block plus the head (bit-exact schedule parity)."""
        e = self._engine
        n = e.n_blocks + 1
        buf = (ctypes.c_int32 * n)()
        e.check(e.lib.cosk_last_schedule(e.h, buf, n), "cosk_last_schedule")
        return tuple(bool(v) for v in buf)

    def read_block(self, index):
        """Last emitted output of block ``index`` as fp32 (N*S, C, V)."""
        e = self._engine
        out = torch.empty((e.n_streams * self._S, self._specs[index].cout, self._V), dtype=torch.float32, device=e.device)
        e.check(e.lib.cosk_read_block(e.h, index, ctypes.c_void_p(out.data_ptr()), self._stream(out)), "cosk_read_block")
        return out

    def state_bytes(self):
        return int(self._engine.lib.cosk_state_bytes(self._engine.h)) if self._engine else 0

    def launch_count(self):
        return int(self._engine.lib.cosk_launch_count(self._engine.h)) if self._engine else 0

    def tensor_core_blocks(self):
        e = self._engine
        return [int(e.lib.cosk_block_uses_tensor_cores(e.h, i)) for i in range(e.n_blocks)]

    def device_error(self):
        e = self._engine
        code = ctypes.c_uint32(0)
        e.check(e.lib.cosk_device_error(e.h, ctypes.byref(code)), "cosk_device_error")
        return int(code.value)

    def knobs(self):
        """The kernel selection of the engine (cosk_describe): runtime knobs and the kernel serving each block."""
        import json

        e = self._engine
        buf = ctypes.create_string_buffer(8192)
        e.check(e.lib.cosk_describe(e.h, buf, len(buf)), "cosk_describe")
        return json.loads(buf.value.decode())

    def trace_read(self, n=24):
        e = self._engine
        buf = (ctypes.c_uint64 * n)()
        e.check(e.lib.cosk_trace_read(e.h, buf, n), "cosk_trace_read")
        return [int(v) for v in buf]

    def profile(self, on):
        e = self._engine
        e.check(e.lib.cosk_profile_enable(e.h, 1 if on else 0), "cosk_profile_enable")

    def profile_read(self, kind, block=-1):
        e = self._engine
        ms, n = ctypes.c_double(0), ctypes.c_int64(0)
        e.check(e.lib.cosk_profile_read(e.h, kind, block, ctypes.byref(ms), ctypes.byref(n)), "cosk_profile_read")
        return float(ms.value), int(n.value)

    # -- stepping -----------------------------------------------------------------------------
    def _out_shape(self, n_streams):
        if self._head:
            return (n_streams, self._classes)
        return (n_streams * self._S, self._specs[-1].cout, self._V)

    def _step(self, x, n_streams, nc_stride):
        e = self._sync(x.device)
        self._ensure_batch(e, (n_streams,) + tuple(x.shape[1:]), n_streams)
        out = torch.empty(self._out_shape(n_streams), dtype=torch.float32, device=x.device)
        em = ctypes.c_int32(0)
        try:
            e.check(e.lib.cosk_step(e.h, ctypes.c_void_p(x.data_ptr()), nc_stride, ctypes.c_void_p(out.data_ptr()),
                                    ctypes.byref(em), self._stream(x)), "cosk_step")
        except CoskError:
            self._shape = None  # the handle latched a failure: the next call re-creates (and zeroes) all state
            raise
        return out if em.value else None

    def _steps(self, x, n_streams, T, shape_key, pad_end=False):
        e = self._sync(x.device)
        self._ensure_batch(e, shape_key, n_streams, T)
        # upper bound on emissions: the last stage can emit at most once per `stride` frames; the end-of-sequence flush
        # adds at most one emission per padded frame of any stage
        max_out = T // self.stride + 1
        if pad_end:
            max_out += self._pad * len(self._specs) + (self.pool_padding if self._head else 0) + 1
        oshape = self._out_shape(n_streams)
        out = torch.empty((max_out,) + oshape, dtype=torch.float32, device=x.device)
        n = ctypes.c_int32(0)
        try:
            e.check(e.lib.cosk_steps_ex(e.h, ctypes.c_void_p(x.data_ptr()), T, ctypes.c_void_p(out.data_ptr()),
                                        int(np.prod(oshape)), max_out, ctypes.byref(n), self._stream(x), 1 if pad_end else 0),
                    "cosk_steps")
        except CoskError:
            self._shape = None
            raise
        if n.value == 0:
            return None
        return out[: n.value]


# ---------------------------------------------------------------------------------------------
# full models
# ---------------------------------------------------------------------------------------------
class CoModelBase(_CoBase):
    """Continual ST-GCN model: data_bn -> 10 blocks -> spatial mean -> sliding mean -> fc
    (CoModelBase.on_init_end, models/base.py:68-122)."""

    PADDING = 4
    STRIDED = True
    ADAPTIVE = False  # AdaptiveGraphConvolution instead of GraphConvolution (CoAGcn)

    @staticmethod
    def configs():
        c = Configs()
        # models/base.py:23-66
        c.add("forward_mode", "clip")
        c.add("predict_after_frames", 0)
        c.add("continual_temporal_fill", "replicate")
        c.add("pool_size", -1)
        c.add("pool_padding", -1)
        # datasets/datasets.py:15-22,73-79 (the keys that shape the model)
        c.add("dataset_name", "dummy_ntu")
        c.add("dataset_input_channels", 3)
        c.add("batch_size", 2)
        c.add("profile_model", False)
        # this implementation
        c.add("kernel_path", "auto")
        c.add("time_chunk", -1)  # frames per launch of forward_steps: -1 auto (see _pick_time_chunk), 1 = step by step
        return c

    @classmethod
    def block_specs(cls, c_in):
        s = 2 if cls.STRIDED else 1
        # models/cost_gcn/cost_gcn.py:30-41, models/cost_gcn_mod/cost_gcn_mod.py:29-40
        return [
            BlockSpec(c_in, 64, 1, residual=False),
            BlockSpec(64, 64), BlockSpec(64, 64), BlockSpec(64, 64),
            BlockSpec(64, 128, s), BlockSpec(128, 128), BlockSpec(128, 128),
            BlockSpec(128, 256, s), BlockSpec(256, 256), BlockSpec(256, 256),
        ]

    def __init__(self, hparams=None, **overrides):
        super().__init__()
        hp = self.configs().default_values()
        if hparams is not None:
            hp.update(vars(hparams) if not isinstance(hparams, dict) else hparams)
        hp.update(overrides)
        self.hparams = AttributeDict(hp)
        classes, graph_fn = DATASETS[self.hparams.dataset_name]
        self.graph = graph_fn()
        c_in = int(self.hparams.dataset_input_channels)
        V, S, T = self.graph.num_node, 2, 300
        self.input_shape = (c_in, T, V, S)
        self.output_shape = (classes,)
        self.num_classes = classes
        specs = self.block_specs(c_in)
        self._setup(specs, self.PADDING, V, S, c_in, classes, True, self.graph.A, self.hparams.kernel_path, self.ADAPTIVE)
        self._time_chunk = int(self.hparams.time_chunk)

        self.data_bn = nn.BatchNorm1d(S * c_in * V)
        _init_bn(self.data_bn, 1)
        self.layers = _Node()
        for i, sp in enumerate(self._specs):
            self.layers.add_module(f"layer{i + 1}", _block_params(sp, self.graph.A, self.PADDING, sp.gconv))
        self.fc = nn.Linear(256, classes)
        nn.init.normal_(self.fc.weight, 0, math.sqrt(2.0 / classes))  # models/utils.py:23-24

        # models/base.py:86-97
        pool_size = int(self.hparams.pool_size)
        if pool_size == -1:
            pool_size = math.ceil((T - self.receptive_field + 2 * self.padding + 1) / self.stride)
        pool_padding = int(self.hparams.pool_padding)
        if pool_padding == -1:
            pool_padding = pool_size - math.ceil((T - self.receptive_field + self.padding + 1) / self.stride)
        self.pool_size, self.pool_padding = pool_size, max(0, pool_padding)
        # The values above are those of the block stack, which is what the reference's pool formulas see
        # (models/base.py:86-96 run before the full module list exists).  Once co.Sequential holds data_bn,
        # blocks, pool and fc, its receptive_field / padding / delay include the pooling window -- and that is
        # what warm_up (models/base.py:155) uses: 449 / 152 / 296 for CoST-GCN, 300 / 0 / 299 for CoST-GCN*.
        self.stack_receptive_field, self.stack_padding = self.receptive_field, self.padding
        self.receptive_field += (self.pool_size - 1) * self.stride
        self.padding += self.pool_padding * self.stride
        self.delay = self.receptive_field - 1 - self.padding
        self.call_mode = "forward_steps" if self.hparams.forward_mode == "frame" else "forward"
        if self.hparams.profile_model and self.hparams.forward_mode == "frame":
            self.input_shape = (c_in, self.stride, V, S)  # models/base.py:135-142
        self.eval()

    def _block_modules(self):
        return [getattr(self.layers, f"layer{i + 1}") for i in range(len(self._specs))]

    # models/base.py:200-227
    def map_state_dict(self, state_dict, strict=True):
        def short(k):
            return k.replace("0.1.", "").replace("0.0.residual", "residual")

        own = list(nn.Module.state_dict(self, keep_vars=True).keys())
        if set(own) - set(state_dict.keys()):
            table = {short(k): k for k in own}
            state_dict = OrderedDict((table[k], v) for k, v in state_dict.items() if strict or k in table)
        return state_dict

    def map_loaded_weights(self, file, loaded_state_dict):
        return self.map_state_dict(loaded_state_dict)

    def validate_attributes(self):
        for i in range(10):
            assert isinstance(getattr(self.layers, f"layer{i + 1}"), nn.Module)

    # models/base.py:144-159
    def warm_up(self, dummy=None, sample=None, *a, **kw):
        if self.hparams.forward_mode == "clip":
            return
        self.clean_state()
        N, C = sample.shape[0], sample.shape[1]
        V, S = self._V, self._S
        frames = self.receptive_field - self.padding - 1
        dev = sample.device if sample.device.type == "cuda" else torch.device("cuda", torch.cuda.current_device())
        data = torch.randn((N, C, frames, V, S), device=dev)
        self.forward_steps(data)

    def forward_step(self, input, update_state=True):
        """input (N, C, V, S) -> logits (N, classes) when a prediction is due, else None
        (models/base.py:183-185; the library's "no output yet" placeholder is None here)."""
        if not update_state:
            raise NotImplementedError("update_state=False is not supported (never used by the reference models)")
        x = self._check_input(input, 4)
        return self._step(x, x.shape[0], self._V * self._S)

    def forward_steps(self, input, pad_end=False, update_state=True):
        """input (N, C, T, V, S) -> (N, classes) for one emission, (N, classes, n) for several, None
        for none (models/base.py:187-190,101).  ``pad_end=True`` (the library's end-of-clip flush, used by the reference's
        tests): every temporal stage is fed its end padding after the clip, so the emissions equal the regular zero-padded
        network's outputs over the whole clip; the state is reset afterwards (the padded frames are not part of the stream)."""
        if not update_state:
            raise NotImplementedError("update_state=False is not supported")
        x = self._check_input(input, 5)
        N, C, T, V, S = x.shape
        out = self._steps(x, N, T, (N, C, V, S), pad_end)
        if out is None:
            return None
        return out[0] if out.shape[0] == 1 else out.permute(1, 2, 0).contiguous()

    def forward(self, input):
        """models/base.py:166-181.  "frame": reset (unless profiling) and step through the clip.
        "clip": the reference runs the same weights as a regular padded network and keeps output 0;
        that first output only depends on the first ``delay + 1`` frames (297 / 300) and no end padding, so it is produced here by stepping a fresh state."""
        if self.hparams.forward_mode == "frame":
            if not self.hparams.profile_model:
                self.clean_state()
        else:
            self.clean_state()
        ret = self.forward_steps(input)
        if ret is not None and ret.dim() == 3:
            ret = ret[:, :, 0]
        return ret


class CoStGcn(CoModelBase):
    """CoST-GCN: "equal" temporal padding, stride 2 at layers 5 and 8 (models/cost_gcn/cost_gcn.py)."""

    PADDING, STRIDED = 4, True


class CoStGcnMod(CoModelBase):
    """CoST-GCN*: no temporal padding, stride 1 everywhere (models/cost_gcn_mod/cost_gcn_mod.py)."""

    PADDING, STRIDED = 0, False


class CoAGcn(CoModelBase):
    """CoA-GCN: the CoST-GCN geometry with ``AdaptiveGraphConvolution`` stepped one frame at a time
    (models/coa_gcn/coa_gcn.py:11-46; the vertex attention of a step sees that step's frame only).

    Only the per-step semantics are implemented: ``forward_step`` / ``forward_steps`` / ``forward`` in
    ``forward_mode="frame"``.  The reference's CLIP forward of this model is a different function -- it runs
    ``AdaptiveGraphConvolution.forward`` on the whole clip, so its softmax attention is taken over all T frames
    (models/a_gcn/a_gcn.py:53-62) -- and is not reproduced by stepping, so ``forward`` in ``"clip"`` mode raises."""

    PADDING, STRIDED, ADAPTIVE = 4, True, True

    def forward(self, input):
        if self.hparams.forward_mode != "frame":
            raise NotImplementedError(
                "CoAGcn implements the continual per-step path only: the reference's clip forward attends over all T frames "
                "(models/a_gcn/a_gcn.py:53-62), which stepping does not reproduce; construct with forward_mode='frame'")
        return super().forward(input)


class CoSTr(CoModelBase):
    """CoS-TR: the CoST-GCN geometry with the spatial self-attention unit ``GcnUnitAttention`` as the graph conv of
    layers 4-10, stepped one frame at a time (models/cos_tr/cos_tr.py:12-47)."""

    PADDING, STRIDED = 4, True

    @classmethod
    def block_specs(cls, c_in):
        specs = super().block_specs(c_in)
        return specs[:3] + [sp._replace(gconv="attention") for sp in specs[3:]]

    def load_state_dict(self, state_dict, strict=True, **kw):
        """CoSTr maps regular S-TR keys by itself when loading (models/cos_tr/cos_tr.py:73-79)."""
        return super().load_state_dict(self.map_state_dict(state_dict, strict), strict=strict, **kw)


# ---------------------------------------------------------------------------------------------
# headless stack of blocks (what the reference's block-level tests build with co.Sequential)
# ---------------------------------------------------------------------------------------------
class CoStack(_CoBase):
    """``co.Sequential(CoSpatioTemporalBlock, ...)`` without data_bn / pooling / fc.
    Children are named "0", "1", ... like ``continual.Sequential`` names them
    (tests/test_cost_gcn.py:288-312 in the reference)."""

    def __init__(self, blocks, padding=4, skeleton="ntu", kernel_path="auto", adaptive=False, time_chunk=-1):
        super().__init__()
        self._time_chunk = int(time_chunk)
        g = _graph.ntu_graph() if skeleton == "ntu" else _graph.kinetics_graph()
        specs = [b if isinstance(b, BlockSpec) else BlockSpec(*b) for b in blocks]
        self._setup(specs, padding, g.num_node, 1, specs[0].cin, 0, False, g.A, kernel_path, adaptive)
        for i, sp in enumerate(self._specs):
            self.add_module(str(i), _block_params(sp, g.A, padding, sp.gconv))
        self.eval()

    def _block_modules(self):
        return [getattr(self, str(i)) for i in range(len(self._specs))]

    def forward_step(self, input):
        """(B, C, V) -> (B, Cout, V) | None."""
        x = self._check_input(input, 3)
        return self._step(x, x.shape[0], self._V)

    def forward_steps(self, input, pad_end=False):
        """(B, C, T, V) -> (B, Cout, n, V) | None.  ``pad_end``: flush every block's temporal end padding after the clip
        (tests/test_cost_gcn.py:67,223,270,325 in the reference), state reset afterwards."""
        x = self._check_input(input, 4)
        B, C, T, V = x.shape
        out = self._steps(x, B, T, (B, C, V), pad_end)
        return None if out is None else out.permute(1, 2, 0, 3).contiguous()
