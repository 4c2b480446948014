"""CPU tests of the boundary: the C-ABI library builds for sm_100a, loads and exports every symbol
include/cosk.h declares; the host mirror has the reference's names, key mapping and geometry; the
host-side BN folding reproduces the oracle; the product path fails loudly without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import continual_skeletons_b200 as cs
from continual_skeletons_b200 import lib as cslib
from continual_skeletons_b200 import model as csmodel
from oracle import regular, weights
from oracle.weights import ArchSpec

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    path = cs.build_library()
    lib = ctypes.CDLL(path)
    header = open(os.path.join(ROOT, "include", "cosk.h")).read()
    declared = set(re.findall(r"\b(cosk_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(cslib.SYMBOLS), declared ^ set(cslib.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    lib.cosk_version.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.cosk_version()


def test_config_struct_matches_header():
    # 12 int32 fields + 16 blocks of 5 int32
    assert ctypes.sizeof(cslib.Config) == 4 * (12 + 5 * cslib.MAX_BLOCKS)
    header = open(os.path.join(ROOT, "include", "cosk.h")).read()
    body = header[header.index("typedef struct {\n  int32_t abi_version"): header.index("} cosk_config;")]
    fields = re.findall(r"int32_t\s+(\w+);", body)
    assert fields == [n for n, _ in cslib.Config._fields_[:-1]]
    assert int(re.search(r"#define COSK_ABI_VERSION (\d+)", header).group(1)) == cslib.ABI_VERSION
    blk = header[header.index("typedef struct {\n  int32_t cin, cout;"): header.index("} cosk_block_cfg;")]
    assert re.findall(r"int32_t\s+([\w, ]+);", blk) == ["cin, cout", "stride", "res_kind", "gconv"]
    assert [n for n, _ in cslib.BlockCfg._fields_] == ["cin", "cout", "stride", "res_kind", "gconv"]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_gpu():
    lib = cs.load_library()
    cfg = cslib.Config()
    cfg.abi_version, cfg.vertices, cfg.persons, cfg.c_in, cfg.n_blocks, cfg.padding = cslib.ABI_VERSION, 25, 1, 4, 1, 4
    cfg.blocks[0].cin, cfg.blocks[0].cout, cfg.blocks[0].stride, cfg.blocks[0].res_kind = 4, 4, 1, 0
    h = ctypes.c_void_p()
    assert lib.cosk_create(ctypes.byref(cfg), ctypes.byref(h)) == -2  # COSK_ERR_CUDA
    assert not h.value
    m = cs.CoStGcn()
    with pytest.raises(cs.CoskError):
        m.forward_step(torch.rand(2, 3, 25, 2))
    with pytest.raises(cs.CoskError):
        m.forward_steps(torch.rand(2, 3, 10, 25, 2))


def test_bad_config_rejected():
    lib = cs.load_library()
    cfg = cslib.Config()
    h = ctypes.c_void_p()
    assert lib.cosk_create(ctypes.byref(cfg), ctypes.byref(h)) == -1  # abi_version 0
    assert lib.cosk_create(None, ctypes.byref(h)) == -1


def test_graph_bit_exact(golden):
    assert np.array_equal(cs.ntu_graph().A, golden["adjacency"]["ntu"])
    assert np.array_equal(cs.kinetics_graph().A, golden["adjacency"]["kinetics"])
    assert cs.ntu_graph().A.dtype == np.float64


@pytest.mark.parametrize("cls,arch_fn,geom", [
    (cs.CoStGcn, weights.cost_gcn_arch, (449, 4, 152, 296, 75, 19)),
    (cs.CoStGcnMod, weights.cost_gcn_mod_arch, (300, 1, 0, 299, 220, 0)),
    (cs.CoAGcn, weights.coa_gcn_arch, (449, 4, 152, 296, 75, 19)),
])
def test_geometry_and_key_mapping(cls, arch_fn, geom):
    m = cls(cls.configs().default_values())
    assert (m.receptive_field, m.stride, m.padding, m.delay, m.pool_size, m.pool_padding) == geom
    arch = arch_fn()  # block stack alone: what the pool formulas of models/base.py:86-96 see
    assert (m.stack_receptive_field, m.stack_padding) == (arch.receptive_field, arch.stack_padding)
    assert m.delay == arch.receptive_field - 1 - arch.stack_padding + (arch.pool_size - 1 - arch.pool_padding) * arch.stack_stride
    assert m.input_shape == (3, 300, 25, 2) and m.output_shape == (60,)
    m.validate_attributes()
    own = list(m.state_dict().keys())
    # nested names of the reference's continual model (SURVEY.md section 3.5)
    assert "layers.layer1.gcn.g_conv.0.weight" in own
    assert "layers.layer2.0.1.tcn.t_conv.weight" in own
    assert "layers.layer5.0.0.residual.bn.running_var" in own
    assert "layers.layer8.0.1.gcn.gcn_residual.1.weight" in own
    sd = weights.make_state_dict(arch_fn(), seed=1, randomize=True)  # regular StGcn keys
    mapped = m.map_state_dict(sd, strict=True)
    assert sorted(mapped.keys()) == sorted(own)
    res = m.load_state_dict(mapped, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    back = m.state_dict()
    assert torch.equal(back["layers.layer5.0.0.residual.t_conv.weight"], sd["layers.layer5.residual.t_conv.weight"])
    # already-continual keys pass through unchanged
    assert list(m.map_state_dict(back).keys()) == own


def test_reference_style_init():
    torch.manual_seed(0)
    m = cs.CoStGcn()
    sd = m.state_dict()
    assert torch.all(sd["layers.layer3.0.1.gcn.bn.weight"] == 1e-6)  # models/base.py:256-257
    assert torch.all(sd["layers.layer3.0.1.gcn.graph_attn"] == 1)
    assert torch.all(sd["layers.layer1.tcn.t_conv.bias"] == 0)
    w = sd["layers.layer9.0.1.tcn.t_conv.weight"]
    assert abs(float(w.std()) - (2.0 / (256 * 9)) ** 0.5) < 2e-3  # kaiming fan_out
    assert not sd["layers.layer3.0.1.gcn.A"].requires_grad


@pytest.mark.parametrize("cin,cout,stride,residual,pad", [(4, 4, 1, True, 4), (2, 4, 2, True, 4), (3, 8, 1, False, 0)])
def test_host_bn_folding_matches_oracle(cin, cout, stride, residual, pad):
    """The folded tensors handed to cosk_load_weights, applied with plain torch ops, reproduce the
    oracle's graph conv and temporal conv (host logic, no GPU)."""
    spec = cs.BlockSpec(cin, cout, stride, residual)
    arch = ArchSpec([weights.BlockSpec(cin, cout, stride, residual)], padding=pad, head=False, block_names=[""])
    sd = weights.make_state_dict(arch, seed=21, randomize=True)
    stack = cs.CoStack([spec], padding=pad)
    prefix = "0." if spec.res_kind == 0 else None
    mapped = {}
    for k, v in sd.items():
        if spec.res_kind == 0:
            mapped["0." + k] = v
        elif k.startswith("residual"):
            mapped["0.0.0." + k] = v
        else:
            mapped["0.0.1." + k] = v
    stack.load_state_dict(mapped, strict=True)
    f = csmodel._folded_block_tensors(stack._block_modules()[0], spec)
    x = weights.make_input((2, cin, 12, 25), seed=22)
    # graph conv with folded tensors
    mix = f["mix"]
    parts = [torch.einsum("bctv,vw->bctw", x, mix[i]) for i in range(3)]
    if cin != cout:
        parts.append(x)
    cat = torch.cat(parts, dim=1)  # (B, K, T, V), K partition-major
    g = torch.relu(torch.einsum("ok,bktv->botv", f["gcn.w"], cat) + f["gcn.b"][None, :, None, None] + (x if cin == cout else 0))
    want = regular.graph_conv(x, sd, "gcn.")
    assert torch.allclose(g, want, atol=2e-6 * max(1.0, float(want.abs().max())))
    # temporal conv (valid, 9 taps, tap-major K) on frames 0..8 -> regular output index 4 - pad... compare unpadded
    wt = f["tcn.w"].view(cout, 9, cout)
    win = want[:, :, 0:9]  # (B, C, 9, V)
    y = torch.einsum("okc,bckv->bov", wt, win) + f["tcn.b"][None, :, None]
    ref = regular.temporal_conv(want, sd, "tcn.", 1, 0)[:, :, 0]
    if spec.res_kind == 2:
        rr = regular.temporal_conv(x[:, :, 4:5], sd, "residual.", 1, 0)[:, :, 0]
        y = y + torch.einsum("oc,bcv->bov", f["res.w"], x[:, :, 4])
        ref = ref + rr
    assert torch.allclose(y, ref, atol=5e-6 * max(1.0, float(ref.abs().max())))


def test_unsupported_arguments():
    m = cs.CoStGcn()
    with pytest.raises(NotImplementedError):
        m.forward_steps(torch.rand(1, 3, 4, 25, 2), update_state=False)
    with pytest.raises(NotImplementedError):
        m.forward_step(torch.rand(1, 3, 25, 2), update_state=False)
    # CoA-GCN implements the per-step path only: its clip forward is a different function in the reference
    # (attention over all T frames, models/a_gcn/a_gcn.py:53-62) and is refused rather than approximated
    a = cs.CoAGcn()
    with pytest.raises(NotImplementedError):
        a(torch.rand(1, 3, 4, 25, 2))
    # no CPU path: host tensors are refused, pad_end or not
    with pytest.raises(cs.CoskError):
        m.forward_steps(torch.rand(1, 3, 4, 25, 2), pad_end=True)


@pytest.mark.parametrize("cls,arch_fn", [(cs.CoStGcn, weights.cost_gcn_arch), (cs.CoStGcnMod, weights.cost_gcn_mod_arch)])
def test_host_schedule_bit_exact_vs_step_oracle(cls, arch_fn):
    """The library's integer bookkeeping (which block fires on which frame, when logits are due),
    run on the host without a GPU, equals the step oracle's trace for 320 frames."""
    from oracle import step

    arch = arch_fn()
    sd = weights.make_state_dict(arch, seed=3)
    ref = step.StepModel(sd, arch)
    T = 320
    x = torch.zeros(1, 3, 25, 2)
    with torch.no_grad():
        for _ in range(T):
            ref.forward_step(x)
    got = cls().simulate_schedule(T)
    assert got == [tuple(f) for f in ref.trace]
    first = [t for t, f in enumerate(got) if f[-1]][0]
    assert first == (296 if cls is cs.CoStGcn else 299)


def test_host_schedule_of_a_strided_stack():
    from oracle import step

    blocks = [weights.BlockSpec(3, 4, 2, True), weights.BlockSpec(4, 4, 1, True), weights.BlockSpec(4, 8, 2, True)]
    for pad in (4, 0):
        arch = ArchSpec(blocks, padding=pad, head=False, block_names=["0.", "1.", "2."])
        sd = weights.make_state_dict(arch, seed=5)
        ref = step.StepModel(sd, arch)
        x = torch.zeros(1, 3, 25)
        with torch.no_grad():
            for _ in range(60):
                ref.forward_step(x)
        stack = cs.CoStack([cs.BlockSpec(b.cin, b.cout, b.stride, b.residual) for b in blocks], padding=pad)
        assert stack.simulate_schedule(60) == [tuple(f) for f in ref.trace]


def test_aggregate_preds_matches_numpy_reduction():
    """scripts/multi_stream_eval.py:33-42: reduce with np.add / np.maximum, equal shapes required."""
    import numpy as np
    import torch

    import continual_skeletons_b200 as cs

    rng = np.random.default_rng(0)
    preds = [rng.standard_normal((6, 60)).astype(np.float32) for _ in range(3)]
    tp = [torch.from_numpy(p) for p in preds]
    np.testing.assert_array_equal(cs.aggregate_preds(tp, "add").numpy(), (preds[0] + preds[1]) + preds[2])
    np.testing.assert_array_equal(cs.aggregate_preds(tp, "max").numpy(), np.maximum(np.maximum(preds[0], preds[1]), preds[2]))
    with pytest.raises(ValueError):
        cs.aggregate_preds([tp[0], tp[1][:3]])
    with pytest.raises(ValueError):
        cs.aggregate_preds(tp, "mean")


def test_coa_gcn_host_model():
    """CoAGcn: the reference's nested key names for the embedding convs (models/a_gcn/a_gcn.py:22-31 under the
    CoSpatioTemporalBlock wrappers), its init (models/utils.py:10-19 with bs = 1; graph_attn = 1 as an additive term),
    the folded tensors of the adaptive layout, and NTU-120 class count (BASELINE configs[2])."""
    torch.manual_seed(0)
    m = cs.CoAGcn({"dataset_name": "ntu120"})
    assert m.num_classes == 120
    assert [m._config().blocks[i].gconv for i in range(10)] == [1] * 10 and cs.CoStGcn()._config().blocks[3].gconv == 0
    sd = m.state_dict()
    assert sd["layers.layer1.gcn.a_conv.0.weight"].shape == (16, 3, 1, 1)
    assert sd["layers.layer10.0.1.gcn.b_conv.2.weight"].shape == (64, 256, 1, 1)
    assert torch.all(sd["layers.layer4.0.1.gcn.a_conv.1.bias"] == 0)
    w = sd["layers.layer9.0.1.gcn.a_conv.0.weight"]
    assert abs(float(w.std()) - (2.0 / 64) ** 0.5) < 2e-2  # kaiming fan_out over inter_c = 64 outputs
    from continual_skeletons_b200 import model as _m

    blk, spec = m.layers.layer5, m._specs[4]
    t = _m._folded_block_tensors(blk, spec)
    gcn = blk._cosk_parts[0]
    assert torch.equal(t["mix"], (gcn.A + gcn.graph_attn).detach().float())
    assert t["att.w"].shape == (6 * 32, 64) and t["att.b"].shape == (6 * 32,)
    assert torch.equal(t["att.w"][32:64], gcn.b_conv[0].weight.detach()[:, :, 0, 0])  # rows: theta_0, phi_0, theta_1, ...
    assert torch.equal(t["att.w"][64:96], gcn.a_conv[1].weight.detach()[:, :, 0, 0])
    with pytest.raises(ValueError):
        cs.CoStack([cs.BlockSpec(2, 2, 1, True)], adaptive=True)  # out_channels // 4 == 0, as in the reference


def test_cos_tr_host_model(golden):
    """CoSTr: the reference's key names for the attention unit (models/s_tr/s_tr.py:352-415 under the block wrappers),
    strict loading of a regular S-TR state_dict, and the folded tensors reproducing the oracle's unit (host logic)."""
    m = cs.CoSTr({"dataset_name": "dummy_kin"})
    assert m.num_classes == 400 and m._V == 18
    assert [m._config().blocks[i].gconv for i in range(10)] == [0, 0, 0] + [2] * 7
    own = list(m.state_dict().keys())
    assert "layers.layer4.0.1.gcn.attention_conv.qkv_conv.weight" in own
    assert "layers.layer5.0.1.gcn.data_bn.running_mean" in own and "layers.layer3.0.1.gcn.g_conv.2.bias" in own
    arch = weights.cos_tr_arch()
    sd = weights.make_state_dict(arch, seed=8, randomize=True)
    res = m.load_state_dict(m.map_state_dict(sd), strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    res = cs.CoSTr({"dataset_name": "dummy_kin"}).load_state_dict(sd, strict=True)  # regular keys are mapped on load (cos_tr.py:73-79)
    assert not res.missing_keys and not res.unexpected_keys
    from continual_skeletons_b200 import model as _m

    blk, spec = m.layers.layer6, m._specs[5]
    t = _m._folded_block_tensors(blk, spec)
    assert t["sa.qkv.w"].shape == (2 * 32 + 128, 128) and t["sa.in_scale"].shape == (128 * 18,) and t["gcn.w"].shape == (128, 128)
    # apply the folded tensors with plain torch ops and compare with the oracle's unit on two frames
    x = weights.make_input((3, 128, 2, 18), seed=5)
    want = regular.graph_conv(x, sd, "layers.layer6.gcn.")
    xn = x * t["sa.in_scale"].view(1, 128, 1, 18) + t["sa.in_shift"].view(1, 128, 1, 18)
    qkv = torch.einsum("oc,bctv->botv", t["sa.qkv.w"], xn) + t["sa.qkv.b"].view(1, -1, 1, 1)
    q, k, v = qkv[:, :32], qkv[:, 32:64], qkv[:, 64:]
    B, T, V = 3, 2, 18
    q, k, v = (z.reshape(B, 8, -1, T, V) for z in (q, k, v))
    w = torch.softmax(torch.einsum("bhdti,bhdtj->bhtij", q, k), dim=-1)
    o = torch.einsum("bhtij,bhdtj->bhdti", w, v).reshape(B, 128, T, V)
    got = torch.relu(torch.einsum("oc,bctv->botv", t["gcn.w"], o) + t["gcn.b"].view(1, -1, 1, 1) + t["sa.skip_scale"].view(1, -1, 1, 1) * x)
    assert torch.allclose(got, want, atol=2e-5 * max(1.0, float(want.abs().max())))


def test_bench_algorithmic_cost_matches_survey_totals():
    """bench.py derives the roofline numerators from the block table; they must reproduce the totals SURVEY.md section
    8(d) states (CoST-GCN 1.408 MB / 57.5 M MACs, CoST-GCN* 3.072 MB / 159.0 M MACs per stream-frame, Kinetics 1.014 MB /
    41.0 M MACs) and the per-block figure of 70.4 kB per skeleton for a 64-channel block step."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    a = bench.algorithmic_cost("cost_gcn", v=25)
    assert abs(a["state"] - 1.408e6) < 1 and abs(a["flops"] / 2 - 57.5e6) < 0.05e6
    b = bench.algorithmic_cost("cost_gcn_mod", v=25)
    assert abs(b["state"] - 3.072e6) < 1 and abs(b["flops"] / 2 - 159.0e6) < 0.05e6
    k = bench.algorithmic_cost("cost_gcn", v=18)
    assert abs(k["state"] - 1.01376e6) < 1 and abs(k["flops"] / 2 - 41.0e6) < 0.05e6
    blk = a["blocks"][1]  # a 64 -> 64 block: 11 frames of 25 x 64 x 4 B per skeleton, two skeletons per stream
    assert blk["gcn_bytes"] + blk["tcn_bytes"] == 2 * 70400


@pytest.mark.parametrize("V,graph_fn", [(25, cs.graph.ntu_graph), (18, cs.graph.kinetics_graph)])
def test_compiled_skeleton_trees_match_the_graph(V, graph_fn):
    """k_tc_gcnt (csrc/tc_gcnt.cuh) contracts the adjacency along a skeleton tree that is fixed at compile time
    (skel_parent<V>): partition 1 must be exactly "vertex <- its parent", partition 2 exactly "parent <- its children",
    partition 0 the identity -- the sparsity of the reference's graph (datasets/graph.py:9-44 with the edge lists of
    datasets/ntu_rgbd.py:3-35 and datasets/kinetics.py:24-46), which graph.py reproduces bit for bit."""
    src = open(os.path.join(ROOT, "continual-skeletons_b200", "csrc", "tc_gcnt.cuh")).read()
    m = re.search(r"skel_parent<%d>\(int w\) \{[^\n]*\n\s*constexpr int p\[%d\] = \{([^}]*)\};" % (V, V), src)
    assert m, "parent table not found"
    parent = [int(t) for t in m.group(1).split(",")]
    assert len(parent) == V and parent.count(-1) == 1
    A = graph_fn().A
    assert A.shape == (3, V, V)
    want1 = np.zeros((V, V), dtype=bool)  # [v, w]: z[w] += A_1[v, w] * y[v], v = parent(w)
    want2 = np.zeros((V, V), dtype=bool)  # [v, w]: v = child, w = parent(v)
    for w, p in enumerate(parent):
        if p >= 0:
            want1[p, w] = True
            want2[w, p] = True
    assert np.array_equal(A[0] != 0, np.eye(V, dtype=bool))
    assert np.array_equal(A[1] != 0, want1)
    assert np.array_equal(A[2] != 0, want2)
    # every vertex reaches the root: the table is a tree, not a forest with a cycle
    root = parent.index(-1)
    for w in range(V):
        seen, v = 0, w
        while v != root:
            v, seen = parent[v], seen + 1
            assert seen <= V


def test_every_launched_kernel_has_a_route_case():
    """Every kernel (and template instantiation) csrc/cosk.cu passes to launch_k is declared covered by a case of the GPU
    route table (tests/route_table.py), except the trace and opt-in variants listed in its EXCLUDED set."""
    import route_table

    launched = route_table.launched_kernels()
    assert "k_tc_gcnt<25,1,128>" in launched and "k_tc_tcn2<256>" in launched, sorted(launched)
    assert route_table.EXCLUDED <= launched, sorted(route_table.EXCLUDED - launched)
    reachable = launched - route_table.EXCLUDED
    covered = route_table.covered()
    assert reachable == covered, {"without a route case": sorted(reachable - covered),
                                  "declared but never launched": sorted(covered - reachable)}
