"""GPU parity tests (run on the B200 box with ``-m gpu``): the CUDA path, called through the C ABI,
against the CPU oracle and the committed golden fixtures.

Tolerances.  The north star asks for max |dlogit| <= 1e-3 with identical argmax at the reference's
random init (logit magnitude <= 16).  State is split-bf16 (hi + lo, ~17 mantissa bits) and the dense
contractions are 3-product bf16 MMAs with fp32 accumulation, so block outputs are compared with a
relative bound of 1e-4 of the tensor's magnitude; at the reference init the logit bound is
the north star's absolute 1e-3 for every model; the randomised-BN stress variant has logits up to ~100 and its
bound is scaled by max|logit| / 16 (the unscaled figures are printed and kept in profiles/r2_parity_report.txt).  The emission schedule (which block
fires on which frame) is integer bookkeeping and must match bit for bit.
"""
import os

import numpy as np
import pytest
import torch

import continual_skeletons_b200 as cs
from oracle import regular, step, weights
from oracle.make_golden import ADAPTIVE_BLOCK_CASES, ATTENTION_BLOCK_CASES, BLOCK_B, BLOCK_CASES, BLOCK_T
from oracle.weights import ArchSpec

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
BLOCK_RTOL = 1e-4


def _rel_err(got, want):
    return float((got - want).abs().max()) / max(1.0, float(want.abs().max()))


def _stack_keys(sd, spec):
    out = {}
    for k, v in sd.items():
        if spec.res_kind == 0:
            out["0." + k] = v
        elif k.startswith("residual"):
            out["0.0.0." + k] = v
        else:
            out["0.0.1." + k] = v
    return out


def _block_setup(idx, rnd, path):
    name, cin, cout, stride, residual, pad = BLOCK_CASES[idx]
    arch = ArchSpec([weights.BlockSpec(cin, cout, stride, residual)], padding=pad, head=False, block_names=[""])
    sd = weights.make_state_dict(arch, seed=1000 + idx, randomize=rnd)
    batch = 1 if name.startswith("wide") else BLOCK_B
    x = weights.make_input((batch, cin, BLOCK_T, 25), seed=2000 + idx)
    spec = cs.BlockSpec(cin, cout, stride, residual)
    stack = cs.CoStack([spec], padding=pad, kernel_path=path)
    stack.load_state_dict(_stack_keys(sd, spec), strict=True)
    return name + ("_rnd" if rnd else ""), arch, sd, x, spec, stack


@pytest.mark.parametrize("path", ["simt", "auto"])
@pytest.mark.parametrize("rnd", [False, True])
@pytest.mark.parametrize("idx", range(len(BLOCK_CASES)))
def test_block_step_vs_golden(golden, idx, rnd, path):
    """Frame-by-frame block output j equals the reference block's clip output j
    (tests/test_cost_gcn.py:71-271, tests/test_st_gcn_mod.py:11-54 in the reference)."""
    key, arch, sd, x, spec, stack = _block_setup(idx, rnd, path)
    target = torch.from_numpy(golden["blocks"][key])
    xd = x.to(DEV)
    first = 8 - arch.padding
    emitted = []
    for t in range(x.shape[2]):
        o = stack.forward_step(xd[:, :, t].contiguous())
        due = t >= first and (t - first) % spec.stride == 0
        assert (o is not None) == due, (key, t)
        if o is not None:
            emitted.append(o.cpu())
    assert stack.device_error() == 0, hex(stack.device_error())
    if path == "auto" and key.startswith("wide"):
        assert stack.tensor_core_blocks() == [3], "wide blocks must run on the tcgen05 kernels"
    for j, o in enumerate(emitted):
        assert _rel_err(o, target[:, :, j]) < BLOCK_RTOL, (key, j, _rel_err(o, target[:, :, j]))
    # forward_steps over the same clip gives the same emissions after a reset
    stack.clean_state()
    ys = stack.forward_steps(xd).cpu()
    assert ys.shape[2] == len(emitted)
    for j, o in enumerate(emitted):
        assert torch.equal(ys[:, :, j], o)


def _load_model(cls, arch_fn, rnd, path="auto"):
    arch = arch_fn()
    sd = weights.make_state_dict(arch, seed=8 if rnd else 7, randomize=rnd)
    m = cls({"dataset_name": "dummy_ntu", "kernel_path": path})
    m.load_state_dict(m.map_state_dict(sd), strict=True)
    return arch, sd, m


@pytest.mark.parametrize("path", ["simt", "auto"])
@pytest.mark.parametrize("rnd", [False, True])
@pytest.mark.parametrize("cls,arch_fn,tag", [
    (cs.CoStGcn, weights.cost_gcn_arch, "cost_gcn"),
    (cs.CoStGcnMod, weights.cost_gcn_mod_arch, "cost_gcn_mod"),
])
def test_model_forward_steps_vs_reference(golden, cls, arch_fn, tag, rnd, path):
    """The north-star gate: forward_steps over (N=2, C=3, T=300, V=25, M=2)."""
    arch, sd, m = _load_model(cls, arch_fn, rnd, path)
    x = weights.make_input((2, 3, 300, 25, 2), seed=11)
    out = m.forward_steps(x.to(DEV))
    assert m.device_error() == 0, hex(m.device_error())
    assert out is not None and tuple(out.shape) == (2, 60)
    out = out.cpu()
    sfx = "_rnd" if rnd else ""
    want = torch.from_numpy(golden[tag][f"{tag}_co_logits{sfx}"])  # made with the reference's blocks
    # reference init: the north-star gate in absolute terms; randomised-BN stress variant: relative to max|logit| / 16
    scale = max(1.0, float(want.abs().max()) / 16.0) if rnd else 1.0
    err = float((out - want).abs().max())
    print(f"\n[parity] {tag} {'randomised' if rnd else 'reference-init'} path={path}: max|d|={err:.3e} max|logit|={float(want.abs().max()):.2f}")
    assert err <= 1e-3 * scale, (tag, rnd, path, err, float(want.abs().max()))
    assert torch.equal(out.argmax(1), want.argmax(1))
    assert torch.equal(torch.topk(out, 3).indices, torch.topk(want, 3).indices)
    if path == "auto":
        tc = m.tensor_core_blocks()
        assert tc[0] == 2 and all(v == 3 for v in tc[1:]), tc


@pytest.mark.parametrize("cls,arch_fn", [(cs.CoStGcn, weights.cost_gcn_arch), (cs.CoStGcnMod, weights.cost_gcn_mod_arch)])
def test_model_schedule_and_blocks_vs_step_oracle(cls, arch_fn):
    """Per frame: emission flags bit-exact against the step oracle; block outputs close."""
    arch, sd, m = _load_model(cls, arch_fn, True)
    T = 120
    x = weights.make_input((2, 3, T, 25, 2), seed=12)
    ref = step.StepModel(sd, arch)
    xd = x.to(DEV)
    with torch.no_grad():
        feats = []
        regular.stack_features(regular.normalise_input(x, sd), sd, arch, feats)
    for t in range(T):
        with torch.no_grad():
            want = ref.forward_step(x[:, :, t])
        got = m.forward_step(xd[:, :, t].contiguous())
        assert m.last_schedule() == ref.trace[-1], t
        assert (got is None) == (want is None)
        if t in (40, 83, 119):
            for i in range(10):
                n_out = sum(1 for f in ref.trace if f[i])
                if n_out:
                    e = _rel_err(m.read_block(i).cpu(), feats[i][:, :, n_out - 1])
                    assert e < 2e-4, (t, i, e)
    assert m.device_error() == 0


def test_state_lifecycle():
    """clean_state reproduces results exactly; a batch-shape change resets the state
    (models/base.py:161-164); streams are independent (replicated streams give identical rows)."""
    arch, sd, m = _load_model(cs.CoStGcnMod, weights.cost_gcn_mod_arch, True)
    T = 100
    x = weights.make_input((2, 3, T, 25, 2), seed=13).to(DEV)
    for t in range(T):
        m.forward_step(x[:, :, t].contiguous())
    a = m.read_block(9).clone()
    m.clean_state()
    for t in range(T):
        m.forward_step(x[:, :, t].contiguous())
    assert torch.equal(a, m.read_block(9))
    # 3 streams now: shape change -> fresh state, stream 2 is a copy of stream 0
    x3 = torch.cat([x, x[:1]], 0)
    for t in range(T):
        m.forward_step(x3[:, :, t].contiguous())
    b = m.read_block(9)
    assert torch.equal(b[:4], a)
    assert torch.equal(b[4:6], a[0:2])


def test_many_streams_replicated():
    """Thousands of streams through the tiled kernels: every replica of a stream must produce
    bit-identical logits (tile -> stream mapping independent of N, SURVEY.md section 8e)."""
    arch, sd, m = _load_model(cs.CoStGcn, weights.cost_gcn_arch, True)
    base = weights.make_input((2, 3, 300, 25, 2), seed=11).to(DEV)
    small = m.forward_steps(base)
    reps = 333  # 666 streams: not a multiple of the 2.5 streams per tile
    big = m.forward_steps(base.repeat(reps, 1, 1, 1, 1))
    assert m.device_error() == 0
    assert tuple(big.shape) == (2 * reps, 60)
    assert torch.equal(big.view(reps, 2, 60), small.unsqueeze(0).expand(reps, 2, 60))


def test_long_run_pool_window_exact():
    """Sliding mean over pool_size entries stays exact over many emissions (fp64 running sum):
    after the window is full, logits must equal those of a fresh run over the last frames only
    when the input is periodic.  Here: constant input -> logits converge to a fixed point and the
    running-sum logits equal a recomputation from block outputs."""
    arch, sd, m = _load_model(cs.CoStGcn, weights.cost_gcn_arch, False)
    frame = weights.make_input((1, 3, 25, 2), seed=14).to(DEV)
    outs = []
    for t in range(1200):
        o = m.forward_step(frame)
        if o is not None:
            outs.append(o.clone())
    # with constant input every layer-10 output is identical once warmed up, so the pooled mean is
    # constant after pool_size further emissions and logits stop changing bit for bit
    assert len(outs) > 150
    assert torch.equal(outs[-1], outs[-2]) and torch.equal(outs[-1], outs[-40])


def _load_stack(stack, sd, blocks):
    mapped = {}
    for k, v in sd.items():
        i, rest = k.split(".", 1)
        spec = blocks[int(i)]
        if spec.res_kind == 0:
            mapped[f"{i}.{rest}"] = v
        elif rest.startswith("residual"):
            mapped[f"{i}.0.0.{rest}"] = v
        else:
            mapped[f"{i}.0.1.{rest}"] = v
    stack.load_state_dict(mapped, strict=True)


@pytest.mark.parametrize("rnd", [False, True])
@pytest.mark.parametrize("skeleton,V,B", [("ntu", 25, 23), ("ntu", 25, 1495), ("kinetics", 18, 23)])
@pytest.mark.parametrize("cin,cout", [(64, 128), (128, 128), (128, 256)])
def test_channel_major_graph_conv(monkeypatch, cin, cout, skeleton, V, B, rnd):
    """k_tc_gcnt (channels on the TMEM lanes, adjacency contraction in registers along the compiled-in skeleton tree):
    selected for the 128/256-channel plain graph convs of both skeletons, equal to the oracle's clip math with distinct
    streams, a phantom second tile in the last pair (odd tile counts), more tile pairs than SMs (B = 1495 -> 299 tiles), unit
    self links (three parts, gcn_residual folded into W_0) and trained ones (four parts) -- and to the token-major kernel."""
    blocks = [weights.BlockSpec(cin, cout, 1, True)]
    arch = ArchSpec(blocks, padding=4, skeleton=skeleton, head=False, block_names=["0."])
    sd = weights.make_state_dict(arch, seed=77 + cin + cout, randomize=rnd)
    T = 12
    x = weights.make_input((B, cin, T, V), seed=78)
    with torch.no_grad():
        target = regular.stack_features(x, sd, arch)
    outs = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("COSK_GCN_T", flag)
        stack = cs.CoStack([cs.BlockSpec(cin, cout, 1, True)], padding=4, skeleton=skeleton)
        _load_stack(stack, sd, blocks)
        out = stack.forward_steps(x.to(DEV))
        assert stack.device_error() == 0
        kernel = stack.knobs()["blocks"][0]["gcn"]
        assert kernel.startswith("k_tc_gcnt<%d>" % (4 if rnd else 3)) if flag == "1" else kernel.startswith("k_tc_gcn<")
        outs[flag] = out.cpu()
    n = outs["1"].shape[2]
    assert n == target.shape[2] - arch.stack_padding // arch.stack_stride
    assert _rel_err(outs["1"], target[:, :, :n]) < BLOCK_RTOL
    assert _rel_err(outs["1"], outs["0"]) < 2e-5  # same products, different fp32 summation order of the mix


@pytest.mark.parametrize("path", ["simt", "auto"])
def test_kinetics_skeleton_stack(path):
    """V = 18 (OpenPose) graph, 7 skeletons = 126 token rows per tile, a strided 3-block stack with every
    residual kind: emitted outputs equal the oracle's clip math; odd stream counts leave a ragged last tile."""
    blocks = [weights.BlockSpec(64, 64, 1, False), weights.BlockSpec(64, 64, 1, True), weights.BlockSpec(64, 128, 2, True)]
    arch = ArchSpec(blocks, padding=4, skeleton="kinetics", head=False, block_names=["0.", "1.", "2."])
    sd = weights.make_state_dict(arch, seed=31, randomize=True)
    B, T = 23, 30  # 23 skeletons -> 4 tiles, the last one partly filled
    x = weights.make_input((B, 64, T, 18), seed=32)
    with torch.no_grad():
        target = regular.stack_features(x, sd, arch)
    stack = cs.CoStack([cs.BlockSpec(b.cin, b.cout, b.stride, b.residual) for b in blocks], padding=4, skeleton="kinetics",
                       kernel_path=path)
    mapped = {}
    for k, v in sd.items():
        i, rest = k.split(".", 1)
        spec = blocks[int(i)]
        if spec.res_kind == 0:
            mapped[f"{i}.{rest}"] = v
        elif rest.startswith("residual"):
            mapped[f"{i}.0.0.{rest}"] = v
        else:
            mapped[f"{i}.0.1.{rest}"] = v
    stack.load_state_dict(mapped, strict=True)
    out = stack.forward_steps(x.to(DEV))
    assert stack.device_error() == 0
    out = out.cpu()
    n = out.shape[2]
    assert n == target.shape[2] - arch.stack_padding // arch.stack_stride
    assert _rel_err(out, target[:, :, :n]) < 2e-4
    if path == "auto":
        assert stack.tensor_core_blocks() == [3, 3, 3]


def test_single_stream_and_step_vs_steps():
    """N = 1 (one partly filled tile): step-by-step emissions equal forward_steps bit for bit, and the
    logits match the oracle."""
    arch, sd, m = _load_model(cs.CoStGcnMod, weights.cost_gcn_mod_arch, False)
    x = weights.make_input((1, 3, 302, 25, 2), seed=15)
    xd = x.to(DEV)
    outs = []
    for t in range(x.shape[2]):
        o = m.forward_step(xd[:, :, t].contiguous())
        if o is not None:
            outs.append(o.clone())
    assert len(outs) == 3  # frames 299, 300, 301
    m.clean_state()
    ys = m.forward_steps(xd)
    assert tuple(ys.shape) == (1, 60, 3)
    for j, o in enumerate(outs):
        assert torch.equal(ys[:, :, j], o)
    ref = step.StepModel(sd, arch)
    with torch.no_grad():
        want = ref.forward_steps(x)
    assert float((ys.cpu() - want).abs().max()) <= 1e-3
    assert torch.equal(ys.cpu().argmax(1), want.argmax(1))
    assert m.device_error() == 0


def test_benchmark_script_semantics():
    """scripts/benchmark_all_ntu60.py: warm-up then one prediction per stream on every timed call of `stride` frames."""
    import importlib.util
    import os

    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts", "benchmark_all_ntu60.py")
    spec = importlib.util.spec_from_file_location("benchmark_all_ntu60", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    for name, frames in (("cost_gcn", 4), ("cost_gcn_mod", 1)):
        r = mod.profile_model(name, 8, 3, "dummy_ntu", torch.device(DEV))
        assert r["frames_per_prediction"] == frames and r["predictions_per_s"] > 0


def test_multi_stream_fusion_on_device():
    """Two lock-stepped models (joint / bone modality): fused logits == sum of the members' own logits."""
    import continual_skeletons_b200 as cs

    torch.manual_seed(3)
    members = [cs.CoStGcn({"dataset_name": "dummy_ntu"}) for _ in range(2)]
    solo = [cs.CoStGcn({"dataset_name": "dummy_ntu"}) for _ in range(2)]
    for m, s in zip(members, solo):
        s.load_state_dict(m.state_dict())
    ens = cs.MultiStream(members, "add")
    x = [torch.randn(2, 3, 300, 25, 2, device=DEV) for _ in range(2)]
    fused = ens.forward_steps(x)
    want = solo[0].forward_steps(x[0]) + solo[1].forward_steps(x[1])
    assert fused is not None and torch.equal(fused, want)
    ens.clean_state()
    assert ens.forward_step([x[0][:, :, 0], x[1][:, :, 0]]) is None


# ---------------------------------------------------------------------------------------------
# CoA-GCN: adaptive graph conv (SURVEY.md section 8(f) item 1)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["simt", "auto"])
@pytest.mark.parametrize("rnd", [False, True])
@pytest.mark.parametrize("idx", range(len(ADAPTIVE_BLOCK_CASES)))
def test_adaptive_block_step_vs_golden(golden, idx, rnd, path):
    """Block with AdaptiveGraphConvolution stepped frame by frame == the reference block with per-frame attention."""
    name, cin, cout, stride, residual, pad = ADAPTIVE_BLOCK_CASES[idx]
    arch = ArchSpec([weights.BlockSpec(cin, cout, stride, residual)], padding=pad, head=False, block_names=[""], graph_conv="adaptive")
    sd = weights.make_state_dict(arch, seed=3000 + idx, randomize=rnd)
    wide = "wide" in name
    x = weights.make_input((1 if wide else BLOCK_B, cin, 14 if wide else BLOCK_T, 25), seed=4000 + idx)
    spec = cs.BlockSpec(cin, cout, stride, residual)
    stack = cs.CoStack([spec], padding=pad, kernel_path=path, adaptive=True)
    stack.load_state_dict(_stack_keys(sd, spec), strict=True)
    target = torch.from_numpy(golden["coa_blocks"][name + ("_rnd" if rnd else "")])
    xd = x.to(DEV)
    emitted = []
    for t in range(x.shape[2]):
        o = stack.forward_step(xd[:, :, t].contiguous())
        due = t >= 8 - pad and (t - (8 - pad)) % stride == 0
        assert (o is not None) == due, (name, t)
        if o is not None:
            emitted.append(o.cpu())
    assert stack.device_error() == 0, hex(stack.device_error())
    assert len(emitted) == (x.shape[2] - (8 - pad) + stride - 1) // stride  # no end padding: a prefix of the clip output
    for j, o in enumerate(emitted):
        assert _rel_err(o, target[:, :, j]) < BLOCK_RTOL, (name, rnd, path, j, _rel_err(o, target[:, :, j]))


@pytest.mark.parametrize("path", ["simt", "auto"])
@pytest.mark.parametrize("rnd", [False, True])
def test_coa_gcn_forward_steps_vs_reference(golden, rnd, path):
    """CoAGcn.forward_steps over (2, 3, 300, 25, 2): one prediction at frame 296, logits as the reference blocks give."""
    arch, sd, m = _load_model(cs.CoAGcn, weights.coa_gcn_arch, rnd, path)
    x = weights.make_input((2, 3, 300, 25, 2), seed=11)
    out = m.forward_steps(x.to(DEV))
    assert m.device_error() == 0, hex(m.device_error())
    assert out is not None and tuple(out.shape) == (2, 60)
    out = out.cpu()
    want = torch.from_numpy(golden["coa_gcn"]["coa_gcn_co_logits" + ("_rnd" if rnd else "")])
    scale = max(1.0, float(want.abs().max()) / 16.0) if rnd else 1.0
    err = float((out - want).abs().max())
    print(f"\n[parity] {'randomised' if rnd else 'reference-init'} path={path}: max|d|={err:.3e} max|logit|={float(want.abs().max()):.2f}")
    assert err <= 1e-3 * scale, (rnd, path, err, float(want.abs().max()))
    assert torch.equal(out.argmax(1), want.argmax(1))


def test_coa_gcn_schedule_and_blocks_vs_step_oracle():
    arch, sd, m = _load_model(cs.CoAGcn, weights.coa_gcn_arch, True)
    T = 60
    x = weights.make_input((2, 3, T, 25, 2), seed=12)
    ref = step.StepModel(sd, arch)
    xd = x.to(DEV)
    with torch.no_grad():
        feats = []
        regular.stack_features(regular.normalise_input(x, sd), sd, arch, feats, per_frame=True)
    for t in range(T):
        with torch.no_grad():
            want = ref.forward_step(x[:, :, t])
        got = m.forward_step(xd[:, :, t].contiguous())
        assert m.last_schedule() == ref.trace[-1], t
        assert (got is None) == (want is None)
        if t in (30, 59):
            for i in range(10):
                n_out = sum(1 for f in ref.trace if f[i])
                if n_out:
                    e = _rel_err(m.read_block(i).cpu(), feats[i][:, :, n_out - 1])
                    assert e < 2e-4, (t, i, e)
    assert m.device_error() == 0


def test_coa_gcn_many_streams_replicated_and_reset():
    """Hundreds of CoA-GCN streams through the tiled attention / dense-mix kernels: replicas of a stream give
    bit-identical logits, and a reset reproduces them exactly."""
    arch, sd, m = _load_model(cs.CoAGcn, weights.coa_gcn_arch, True)
    base = weights.make_input((2, 3, 300, 25, 2), seed=11).to(DEV)
    small = m.forward_steps(base)
    assert m.tensor_core_blocks() == [2] + [3] * 9
    reps = 111  # 222 streams: not a multiple of the 2.5 streams per tile
    big = m.forward_steps(base.repeat(reps, 1, 1, 1, 1))
    assert m.device_error() == 0
    assert tuple(big.shape) == (2 * reps, 60)
    assert torch.equal(big.view(reps, 2, 60), small.unsqueeze(0).expand(reps, 2, 60))
    m.clean_state()
    assert torch.equal(m.forward_steps(base.repeat(reps, 1, 1, 1, 1)), big)


@pytest.mark.parametrize("path", ["simt", "auto"])
def test_adaptive_kinetics_skeleton_stack(path):
    """Adaptive blocks on the 18-joint Kinetics graph (7 skeletons per 126-row tile) against the step oracle."""
    blocks = [weights.BlockSpec(64, 64, 1, True), weights.BlockSpec(64, 128, 2, True)]
    arch = ArchSpec(blocks, padding=4, skeleton="kinetics", head=False, block_names=["0.", "1."], graph_conv="adaptive")
    sd = weights.make_state_dict(arch, seed=61, randomize=True)
    x = weights.make_input((9, 64, 30, 18), seed=62)
    stack = cs.CoStack([cs.BlockSpec(64, 64, 1, True), cs.BlockSpec(64, 128, 2, True)], padding=4, skeleton="kinetics",
                       kernel_path=path, adaptive=True)
    mapped = {}
    for k, v in sd.items():
        i, rest = k.split(".", 1)
        mapped[f"{i}.0.0.{rest}" if rest.startswith("residual") else f"{i}.0.1.{rest}"] = v
    stack.load_state_dict(mapped, strict=True)
    want = step.StepModel(sd, arch).forward_steps(x)
    got = stack.forward_steps(x.to(DEV))
    assert stack.device_error() == 0
    assert got is not None and tuple(got.shape) == tuple(want.shape)
    assert _rel_err(got.cpu(), want) < BLOCK_RTOL, _rel_err(got.cpu(), want)
    if path == "auto":
        assert stack.tensor_core_blocks() == [3, 3]


@pytest.mark.skipif(os.environ.get("COSK_TEST_UNVERIFIED") != "1" or os.environ.get("COSK_WITH_AGCNT") != "1",
                    reason="k_tc_agcnt has not run on hardware yet (written after the round's GPU budget was spent): not in the default "
                           "build; COSK_WITH_AGCNT=1 COSK_TEST_UNVERIFIED=1 builds and tests it")
@pytest.mark.parametrize("skeleton,V,B", [("ntu", 25, 23), ("ntu", 25, 745), ("kinetics", 18, 23)])
@pytest.mark.parametrize("cin,cout", [(64, 128), (128, 128), (128, 256)])
def test_channel_major_adaptive_graph_conv(monkeypatch, cin, cout, skeleton, V, B):
    """k_tc_agcnt (adaptive graph conv, dense per-skeleton mix with the channels on the TMEM lanes and the mixing rows broadcast
    from shared memory): selected for the 128/256-channel adaptive blocks, equal to the step oracle on distinct streams
    (ragged last tile; B = 745 -> 149 tiles, more than SMs) and to the token-major kernel k_tc_agcn."""
    blocks = [weights.BlockSpec(cin, cout, 1, True)]
    arch = ArchSpec(blocks, padding=4, skeleton=skeleton, head=False, block_names=["0."], graph_conv="adaptive")
    sd = weights.make_state_dict(arch, seed=91 + cin + cout, randomize=True)
    T = 11
    x = weights.make_input((B, cin, T, V), seed=92)
    want = step.StepModel(sd, arch).forward_steps(x)
    mapped = {}
    for k, v in sd.items():
        i, rest = k.split(".", 1)
        mapped[f"{i}.0.0.{rest}" if rest.startswith("residual") else f"{i}.0.1.{rest}"] = v
    outs = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("COSK_AGCN_T", flag)
        stack = cs.CoStack([cs.BlockSpec(cin, cout, 1, True)], padding=4, skeleton=skeleton, adaptive=True)
        stack.load_state_dict(mapped, strict=True)
        out = stack.forward_steps(x.to(DEV))
        assert stack.device_error() == 0
        kernel = stack.knobs()["blocks"][0]["gcn"]
        assert kernel.endswith("k_tc_agcnt" if flag == "1" else "k_tc_agcn"), kernel
        outs[flag] = out.cpu()
    assert tuple(outs["1"].shape) == tuple(want.shape)
    assert _rel_err(outs["1"], want) < BLOCK_RTOL
    assert _rel_err(outs["1"], outs["0"]) < 2e-5


@pytest.mark.parametrize("cls,arch_fn,tag", [
    (cs.CoStGcn, weights.cost_gcn_arch, "cost_gcn"),
    (cs.CoStGcnMod, weights.cost_gcn_mod_arch, "cost_gcn_mod"),
    (cs.CoAGcn, weights.coa_gcn_arch, "coa_gcn"),
])
def test_full_size_4096_streams_replica_property(golden, cls, arch_fn, tag):
    """BASELINE's full size (4096 concurrent streams per GPU) through a size-independent property: the 2-stream
    parity clip replicated 2048 times must give, for every replica, bit-identical logits -- and those must be the
    logits the 2-stream run gives, which are checked against the reference-block fixture."""
    arch, sd, m = _load_model(cls, arch_fn, False)
    base = weights.make_input((2, 3, 300, 25, 2), seed=11).to(DEV)
    small = m.forward_steps(base)
    want = torch.from_numpy(golden[tag][f"{tag}_co_logits"])
    assert float((small.cpu() - want).abs().max()) <= 1e-3
    reps = 2048
    big = m.forward_steps(base.unsqueeze(0).expand(reps, 2, 3, 300, 25, 2).reshape(2 * reps, 3, 300, 25, 2))
    assert m.device_error() == 0
    assert tuple(big.shape) == (2 * reps, 60)
    assert torch.equal(big.view(reps, 2, 60), small.unsqueeze(0).expand(reps, 2, 60))


# ---------------------------------------------------------------------------------------------
# CoS-TR: spatial self-attention unit (SURVEY.md section 8(f) item 2)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["simt", "auto"])
@pytest.mark.parametrize("rnd", [False, True])
@pytest.mark.parametrize("idx", range(len(ATTENTION_BLOCK_CASES)))
def test_attention_block_step_vs_golden(golden, idx, rnd, path):
    """Block with GcnUnitAttention stepped frame by frame == the reference's block on the NTU / Kinetics graphs."""
    name, cin, cout, stride, residual, pad, skel = ATTENTION_BLOCK_CASES[idx]
    arch = ArchSpec([weights.BlockSpec(cin, cout, stride, residual, gconv="attention")], padding=pad, head=False, block_names=[""], skeleton=skel)
    sd = weights.make_state_dict(arch, seed=5000 + idx, randomize=rnd)
    wide = "wide" in name
    x = weights.make_input((1 if wide else BLOCK_B, cin, 14 if wide else BLOCK_T, arch.vertices), seed=6000 + idx)
    spec = cs.BlockSpec(cin, cout, stride, residual, "attention")
    stack = cs.CoStack([spec], padding=pad, skeleton=skel, kernel_path=path)
    stack.load_state_dict(_stack_keys(sd, spec), strict=True)
    target = torch.from_numpy(golden["cos_blocks"][name + ("_rnd" if rnd else "")])
    xd = x.to(DEV)
    emitted = []
    for t in range(x.shape[2]):
        o = stack.forward_step(xd[:, :, t].contiguous())
        due = t >= 8 - pad and (t - (8 - pad)) % stride == 0
        assert (o is not None) == due, (name, t)
        if o is not None:
            emitted.append(o.cpu())
    assert stack.device_error() == 0, hex(stack.device_error())
    assert len(emitted) == (x.shape[2] - (8 - pad) + stride - 1) // stride
    for j, o in enumerate(emitted):
        assert _rel_err(o, target[:, :, j]) < BLOCK_RTOL, (name, rnd, path, j, _rel_err(o, target[:, :, j]))
    if path == "auto" and wide:
        assert stack.tensor_core_blocks() == [3]


def _load_cos_tr(rnd, path="auto"):
    arch = weights.cos_tr_arch()
    sd = weights.make_state_dict(arch, seed=8 if rnd else 7, randomize=rnd)
    m = cs.CoSTr({"dataset_name": "dummy_kin", "kernel_path": path})
    m.load_state_dict(m.map_state_dict(sd), strict=True)
    return arch, sd, m


@pytest.mark.parametrize("path", ["simt", "auto"])
@pytest.mark.parametrize("rnd", [False, True])
def test_cos_tr_forward_steps_vs_reference(golden, rnd, path):
    """CoSTr.forward_steps over (2, 3, 300, 18, 2) (Kinetics skeleton, 400 classes): logits as the reference blocks give."""
    arch, sd, m = _load_cos_tr(rnd, path)
    x = weights.make_input((2, 3, 300, 18, 2), seed=11)
    out = m.forward_steps(x.to(DEV))
    assert m.device_error() == 0, hex(m.device_error())
    assert out is not None and tuple(out.shape) == (2, 400)
    out = out.cpu()
    want = torch.from_numpy(golden["cos_tr"]["cos_tr_co_logits" + ("_rnd" if rnd else "")])
    scale = max(1.0, float(want.abs().max()) / 16.0) if rnd else 1.0
    err = float((out - want).abs().max())
    print(f"\n[parity] {'randomised' if rnd else 'reference-init'} path={path}: max|d|={err:.3e} max|logit|={float(want.abs().max()):.2f}")
    assert err <= 1e-3 * scale, (rnd, path, err, float(want.abs().max()))
    assert torch.equal(out.argmax(1), want.argmax(1))
    if path == "auto":
        assert m.tensor_core_blocks() == [2] + [3] * 9


def test_cos_tr_schedule_and_replicas():
    """Per-frame emission flags bit-exact against the step oracle; replicated streams give bit-identical logits."""
    arch, sd, m = _load_cos_tr(True)
    T = 40
    x = weights.make_input((2, 3, T, 18, 2), seed=12)
    ref = step.StepModel(sd, arch)
    xd = x.to(DEV)
    for t in range(T):
        with torch.no_grad():
            want = ref.forward_step(x[:, :, t])
        got = m.forward_step(xd[:, :, t].contiguous())
        assert m.last_schedule() == ref.trace[-1], t
        assert (got is None) == (want is None)
    base = weights.make_input((2, 3, 300, 18, 2), seed=11).to(DEV)
    m.clean_state()  # forward_steps continues from the current state (models/base.py:187-190)
    small = m.forward_steps(base)
    reps = 75  # 150 streams x 2 persons = 300 skeletons: not a multiple of the 7 skeletons per tile
    big = m.forward_steps(base.repeat(reps, 1, 1, 1, 1))
    assert m.device_error() == 0
    assert torch.equal(big.view(reps, 2, 400), small.unsqueeze(0).expand(reps, 2, 400))


@pytest.mark.parametrize("mode", ["clip", "frame"])
def test_forward_call_modes(golden, mode):
    """CoModelBase.forward (models/base.py:166-181): in "clip" mode the first prediction of the padded regular
    network, in "frame" mode a reset followed by forward_steps -- both equal the reference-block fixture; with
    profile_model the state is kept between calls and warm_up makes every `stride`-frame call yield a prediction."""
    arch = weights.cost_gcn_arch()
    sd = weights.make_state_dict(arch, seed=7, randomize=False)
    m = cs.CoStGcn({"dataset_name": "dummy_ntu", "forward_mode": mode})
    m.load_state_dict(m.map_state_dict(sd), strict=True)
    assert m.call_mode == ("forward_steps" if mode == "frame" else "forward")
    x = weights.make_input((2, 3, 300, 25, 2), seed=11).to(DEV)
    want = torch.from_numpy(golden["cost_gcn"]["cost_gcn_co_logits"])
    for _ in range(2):  # a second call starts from a clean state again
        out = m(x)
        assert tuple(out.shape) == (2, 60)
        assert float((out.cpu() - want).abs().max()) <= 1e-3
    if mode == "frame":
        p = cs.CoStGcn({"dataset_name": "dummy_ntu", "forward_mode": "frame", "profile_model": True})
        assert p.input_shape == (3, p.stride, 25, 2)
        sample = torch.rand((2,) + p.input_shape, device=DEV)
        p.warm_up(None, sample)
        for _ in range(3):
            o = p(sample)
            assert o is not None and tuple(o.shape) == (2, 60)


@pytest.mark.parametrize("n_streams", [1, 5])
@pytest.mark.parametrize("which", ["coa_gcn", "cos_tr"])
def test_widened_models_ragged_tiles(which, n_streams):
    """Odd stream counts (1 and 5 streams: a single partly filled tile, and skeletons that straddle tiles) through the
    attention / dense-mix kernels: every block's latest output against the step oracle's clip-layout features."""
    if which == "coa_gcn":
        arch, sd, m = _load_model(cs.CoAGcn, weights.coa_gcn_arch, True)
        V = 25
    else:
        arch, sd, m = _load_cos_tr(True)
        V = 18
    T = 34
    x = weights.make_input((n_streams, 3, T, V, 2), seed=21)
    with torch.no_grad():
        feats = []
        regular.stack_features(regular.normalise_input(x, sd), sd, arch, feats, per_frame=True)
    ref = step.StepModel(sd, arch)
    xd = x.to(DEV)
    for t in range(T):
        with torch.no_grad():
            ref.forward_step(x[:, :, t])
        m.forward_step(xd[:, :, t].contiguous())
        assert m.last_schedule() == ref.trace[-1], t
    assert m.device_error() == 0
    for i in range(10):
        n_out = sum(1 for f in ref.trace if f[i])
        if n_out:
            e = _rel_err(m.read_block(i).cpu(), feats[i][:, :, n_out - 1])
            assert e < 2e-4, (which, n_streams, i, e)


# ---------------------------------------------------------------------------------------------
# forward_steps(pad_end=True): the relations of the reference's own tests that flush the end padding
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["simt", "auto"])
@pytest.mark.parametrize("rnd", [False, True])
@pytest.mark.parametrize("idx", range(len(BLOCK_CASES)))
def test_block_forward_steps_pad_end_equals_whole_clip(golden, idx, rnd, path):
    """``co.forward_steps(sample, pad_end=True) == reg(sample)`` for every block kind
    (tests/test_cost_gcn.py:67-68,223-224,270,325 in the reference): with the end padding flushed the emissions are the
    regular zero-padded block's outputs over the WHOLE clip, not just the prefix stepping alone can produce."""
    key, arch, sd, x, spec, stack = _block_setup(idx, rnd, path)
    target = torch.from_numpy(golden["blocks"][key])
    xd = x.to(DEV)
    prefix = stack.forward_steps(xd).cpu()  # pad_end=False: target[:, :, :-delay] (tests/test_cost_gcn.py:219-220)
    assert stack.device_error() == 0
    n_prefix = prefix.shape[2]
    assert n_prefix == target.shape[2] - arch.padding // spec.stride or arch.padding == 0
    stack.clean_state()
    full = stack.forward_steps(xd, pad_end=True).cpu()
    assert stack.device_error() == 0
    assert tuple(full.shape) == tuple(target.shape), (key, tuple(full.shape), tuple(target.shape))
    assert _rel_err(full, target) < BLOCK_RTOL, (key, _rel_err(full, target))
    assert torch.equal(full[:, :, :n_prefix], prefix)
    # the padded frames are not part of the stream: the state starts over afterwards
    again = stack.forward_steps(xd).cpu()
    assert torch.equal(again, prefix)


@pytest.mark.parametrize("path", ["simt", "auto"])
def test_strided_three_block_stack_pad_end(path):
    """tests/test_cost_gcn.py:273-326 in the reference: co.Sequential of three blocks (no residual, identity residual,
    strided conv residual), ``forward_steps(pad_end=True)`` equals the regular stack on the clip -- here also with 64 / 128
    channels so that the fused and tensor-core kernels take the flush path."""
    for cin, cout in ((2, 4), (64, 128)):
        blocks = [weights.BlockSpec(cin, cin, 1, False), weights.BlockSpec(cin, cin, 1, True), weights.BlockSpec(cin, cout, 2, True)]
        arch = ArchSpec(blocks, padding=4, head=False, block_names=["0.", "1.", "2."])
        sd = weights.make_state_dict(arch, seed=71, randomize=True)
        x = weights.make_input((3, cin, 21, 25), seed=72)
        with torch.no_grad():
            target = regular.stack_features(x, sd, arch)
        stack = cs.CoStack([cs.BlockSpec(b.cin, b.cout, b.stride, b.residual) for b in blocks], padding=4, kernel_path=path)
        mapped = {}
        for k, v in sd.items():
            i, rest = k.split(".", 1)
            kind = blocks[int(i)].res_kind
            mapped[f"{i}.{rest}" if kind == 0 else (f"{i}.0.0.{rest}" if rest.startswith("residual") else f"{i}.0.1.{rest}")] = v
        stack.load_state_dict(mapped, strict=True)
        out = stack.forward_steps(x.to(DEV), pad_end=True)
        assert stack.device_error() == 0
        assert tuple(out.shape) == tuple(target.shape), (tuple(out.shape), tuple(target.shape))
        assert _rel_err(out.cpu(), target) < 2e-4, _rel_err(out.cpu(), target)


@pytest.mark.parametrize("cls,arch_fn,tag", [
    (cs.CoStGcn, weights.cost_gcn_arch, "cost_gcn"),
    (cs.CoStGcnMod, weights.cost_gcn_mod_arch, "cost_gcn_mod"),
])
def test_model_forward_steps_pad_end_equals_clip_network(cls, arch_fn, tag):
    """Whole model: with the end padding of every block and of the pooling window flushed, forward_steps returns the
    regular network's full output sequence (co.Sequential.forward of models/base.py:166-181 before the [:, :, 0] cut)."""
    arch, sd, m = _load_model(cls, arch_fn, True)
    x = weights.make_input((2, 3, 300, 25, 2), seed=11)
    with torch.no_grad():
        h = regular.pooled_sequence(x, sd, arch)
        h = torch.nn.functional.avg_pool1d(h, arch.pool_size, stride=1, padding=arch.pool_padding)
        want = torch.einsum("kc,nct->nkt", sd["fc.weight"], h) + sd["fc.bias"][None, :, None]
    got = m.forward_steps(x.to(DEV), pad_end=True)
    assert m.device_error() == 0
    if want.shape[2] == 1:
        want = want[:, :, 0]
    assert tuple(got.shape) == tuple(want.shape), (tag, tuple(got.shape), tuple(want.shape))
    scale = max(1.0, float(want.abs().max()) / 16.0)
    assert float((got.cpu() - want).abs().max()) <= 1e-3 * scale
    assert torch.equal(got.cpu().argmax(1), want.argmax(1))
