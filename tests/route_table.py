"""The route table of tests/test_gpu_routes.py and the kernels it declares covered.

Shared by the GPU route tests and by the CPU test in tests/test_boundary_cpu.py that matches the declared kernels with
every kernel ``launch_k`` can reach in csrc/cosk.cu: a kernel or instantiation added to the dispatcher without a route
case fails the CPU suite.  Kernel names are written as in cosk.cu with the spaces removed, e.g. ``k_tc_gcnt<25,1,128>``.
"""
import os
import re
from collections import namedtuple

import numpy as np
import torch

from oracle import graphs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COSK_CU = os.path.join(ROOT, "continual-skeletons_b200", "csrc", "cosk.cu")

SPT = {"ntu": 5, "kinetics": 7}  # skeletons per 128-row token tile


# --- adjacency variants: (A, graph_attn) of the graph conv, both (3, V, V) -------------------------------------
def _tree(skel):
    """(child, parent) pairs of the skeleton, 0-based."""
    return graphs.SKELETONS[skel][1]


def adjacency(variant, skel, rng):
    A = graphs.adjacency(skel).astype(np.float32)
    V = A.shape[1]
    ga = np.ones_like(A)
    if variant == "ref":  # reference init: unit self links, folded three-part weights
        pass
    elif variant == "signed":  # signed coefficients, four parts
        ga = rng.uniform(-1.5, 1.5, size=A.shape).astype(np.float32)
    elif variant == "pruned":  # tree edges and one self link exactly zero: still the tree's sparsity (or less)
        for child, parent in _tree(skel)[::3]:
            ga[1, parent, child] = 0.0
            ga[2, child, parent] = 0.0
        ga[0, 3, 3] = 0.0
    elif variant == "extra_edge":  # one non-tree edge in partition 1
        child, parent = _tree(skel)[0]
        other = next(v for v in range(V) if A[1, v, child] == 0 and v != child)
        A[1, other, child] = 0.25
    elif variant == "src7":  # a vertex with 7 sources in partitions 1 + 2 (> kMixSlots)
        w = 0
        for v in [u for u in range(V) if u != w][:7]:
            A[2, v, w] = 0.1 + 0.01 * v
        A[1, :, w] = 0.0
    elif variant == "src5_p2":  # a vertex with 5 sources in partition 2 (> kPartSrcMax) and at most 6 in 1 + 2
        w = 0
        A[2, :, w] = 0.0
        for v in [u for u in range(V) if u != w][:5]:
            A[2, v, w] = 0.2
        A[1, :, w] = 0.0
    elif variant == "extra_edge_signed":  # off the tree and no unit self links: four-part token-major graph conv
        A, _ = adjacency("extra_edge", skel, rng)
        return A, adjacency("signed", skel, rng)[1]
    elif variant == "offdiag0":  # partition 0 not diagonal
        A[0, 1, 2] = 0.3
    elif variant == "zero":
        A[:] = 0.0
    else:
        raise ValueError(variant)
    return torch.from_numpy(A), torch.from_numpy(ga)


# --- skeleton counts -----------------------------------------------------------------------------------------------
def wave(tiles_per_item, ctas_per_item, waves, offset):
    """Skeleton count whose grid has ``waves`` full waves of work items plus ``offset`` (a launcher runs at most one CTA
    per SM; a work item is ``tiles_per_item`` token tiles on ``ctas_per_item`` CTAs), with a ragged last tile.  With two
    tiles per item the tile count is odd, so the last item has a phantom tile."""
    return ("wave", tiles_per_item, ctas_per_item, waves, offset)


def skeletons(n, skel, sms):
    if isinstance(n, int):
        return n
    _, per_item, ctas, waves, offset = n
    items = waves * (sms // ctas) + offset
    tiles = per_item * items - (per_item - 1)
    return tiles * SPT[skel] - 2


# --- what the GPU tests check ----------------------------------------------------------------------------------------
def picked(B, skel, sms):
    """Skeletons the oracle checks: all of them at small counts, else the first and last and both sides of every wave
    boundary of the launchers' grids (work items of one tile or of a tile pair, one or two CTAs each)."""
    if B <= 64:
        return list(range(B))
    spt = SPT[skel]
    pick = {0, 1, B - 2, B - 1}
    for tiles in {j * (sms // 2) for j in range(1, 9)} | {j * sms for j in range(1, 5)}:
        for s in (tiles * spt - 1, tiles * spt):
            if 0 <= s < B:
                pick.add(s)
    return sorted(pick)


def signed_coordinates(rng, shape, skel, channel_dim=1):
    """Skeleton coordinates in metres: signed x, y, z in [-2, 4); on Kinetics (x, y, confidence in [0, 1))."""
    x = torch.from_numpy(rng.uniform(-2.0, 4.0, size=shape).astype(np.float32))
    if skel == "kinetics":
        conf = x.narrow(channel_dim, 2, 1)
        conf.copy_(torch.from_numpy(rng.uniform(0.0, 1.0, size=tuple(conf.shape)).astype(np.float32)))
    return x


# --- the table -----------------------------------------------------------------------------------------------------
# shape: (cin, cout, stride, residual, gconv); route: the knobs() entry of the block ({"block": prefix} for the one-kernel
# block step, else {"gcn": prefix, "tcn": exact name}); batched: forward_steps walks the stack time-batched; covers: the
# kernels the case launches besides k_input and k_read_block, which every headless stack step launches.
Case = namedtuple("Case", "skel shape adj n route batched covers path")


def _route(gcn=None, tcn=None, block=None):
    return {"block": block} if block else {"gcn": gcn, "tcn": tcn}


def _c(skel, shape, adj, n, route, batched, covers, path="auto"):
    return Case(skel, shape, adj, n, route, batched, tuple(covers) + ("k_input", "k_read_block"), path)


_B64 = _route(block="k_tc_block64")
# the time-batched walk runs a fused 64 -> 64 block as graph conv + temporal conv launches
_B64_COVERS = ("k_tc_block64", "k_tc_tcn<64>")

ROUTES = {
    # 64 -> 64 identity blocks: one kernel per step while every partition-1/2 row has <= 4 sources
    "block64_ref": _c("ntu", (64, 64, 1, True, ""), "ref", 7, _B64, True, _B64_COVERS + ("k_tc_gcn<3,1,false>",)),
    "block64_signed_kin": _c("kinetics", (64, 64, 1, True, ""), "signed", 9, _B64, True, _B64_COVERS + ("k_tc_gcn<4,1,false>",)),
    "block64_zero": _c("ntu", (64, 64, 1, True, ""), "zero", 3, _B64, True, _B64_COVERS + ("k_tc_gcn<4,1,false>",)),
    "block64_wave_short": _c("ntu", (64, 64, 1, True, ""), "ref", wave(1, 1, 1, -1), _B64, True, _B64_COVERS),
    "block64_wave": _c("ntu", (64, 64, 1, True, ""), "ref", wave(1, 1, 1, 0), _B64, True, _B64_COVERS),
    "block64_wave_over": _c("ntu", (64, 64, 1, True, ""), "ref", wave(1, 1, 1, 1), _B64, True, _B64_COVERS),
    "block64_two_waves": _c("ntu", (64, 64, 1, True, ""), "ref", wave(1, 1, 2, 3), _B64, True, _B64_COVERS),
    "gcn3_src5": _c("ntu", (64, 64, 1, True, ""), "src5_p2", 7, _route("k_tc_gcn<3>", "k_tc_tcn<64>"), True,
                    ("k_tc_gcn<3,1,false>", "k_tc_tcn<64>")),
    "gcn3_src5_wave_over": _c("ntu", (64, 64, 1, True, ""), "src5_p2", wave(1, 1, 1, 1), _route("k_tc_gcn<3>", "k_tc_tcn<64>"),
                              True, ("k_tc_gcn<3,1,false>", "k_tc_tcn<64>")),
    "gcn3_src5_two_waves": _c("ntu", (64, 64, 1, True, ""), "src5_p2", wave(1, 1, 2, 3), _route("k_tc_gcn<3>", "k_tc_tcn<64>"),
                              True, ("k_tc_gcn<3,1,false>", "k_tc_tcn<64>")),
    "simt_src7": _c("ntu", (64, 64, 1, True, ""), "src7", 7, _route("k_gcn_simt", "k_tc_tcn<64>"), False,
                    ("k_gcn_simt", "k_tc_tcn<64>")),
    "simt_offdiag0": _c("ntu", (64, 128, 1, True, ""), "offdiag0", 7, _route("k_gcn_simt", "k_tc_tcn2<128>"), False,
                        ("k_gcn_simt", "k_tc_tcn2<128>")),
    "simt_path": _c("ntu", (64, 128, 2, True, ""), "ref", 7, _route("k_gcn_simt", "k_tcn_simt"), False,
                    ("k_gcn_simt", "k_tcn_simt"), path="simt"),
    # channel-major graph conv on the skeleton tree
    "gcnt3_64_128_s2": _c("ntu", (64, 128, 2, True, ""), "ref", 3, _route("k_tc_gcnt<3>", "k_tc_tcn<128>"), True,
                          ("k_tc_gcnt<25,1,128>", "k_tc_tcn<128>")),
    "gcnt4_128_pruned": _c("ntu", (128, 128, 1, True, ""), "pruned", 12, _route("k_tc_gcnt<4>", "k_tc_tcn2<128>"), True,
                           ("k_tc_gcnt<25,2,128>", "k_tc_tcn2<128>")),
    "gcnt4_128_zero": _c("ntu", (128, 128, 1, True, ""), "zero", 7, _route("k_tc_gcnt<4>", "k_tc_tcn2<128>"), True,
                         ("k_tc_gcnt<25,2,128>", "k_tc_tcn2<128>")),
    "gcnt4_128_256_signed": _c("ntu", (128, 256, 2, True, ""), "signed", 11, _route("k_tc_gcnt<4>", "k_tc_tcn2<256>"), True,
                               ("k_tc_gcnt<25,2,256>", "k_tc_tcn2<256>")),
    "gcnt3_kin_64_128": _c("kinetics", (64, 128, 1, True, ""), "ref", 9, _route("k_tc_gcnt<3>", "k_tc_tcn2<128>"), True,
                           ("k_tc_gcnt<18,1,128>", "k_tc_tcn2<128>")),
    "gcnt3_kin_128_128": _c("kinetics", (128, 128, 1, True, ""), "ref", 9, _route("k_tc_gcnt<3>", "k_tc_tcn2<128>"), True,
                            ("k_tc_gcnt<18,2,128>", "k_tc_tcn2<128>")),
    "gcnt3_kin_128_256": _c("kinetics", (128, 256, 2, True, ""), "ref", 16, _route("k_tc_gcnt<3>", "k_tc_tcn2<256>"), True,
                            ("k_tc_gcnt<18,2,256>", "k_tc_tcn2<256>")),
    # work items of k_tc_gcnt are tile pairs, one CTA each; k_tc_tcn2 runs a pair on two CTAs
    "gcnt_pairs_wave_short": _c("ntu", (128, 128, 1, True, ""), "ref", wave(2, 1, 1, -1), _route("k_tc_gcnt<3>", "k_tc_tcn2<128>"),
                                True, ("k_tc_gcnt<25,2,128>", "k_tc_tcn2<128>")),
    "gcnt_pairs_wave": _c("ntu", (128, 128, 1, True, ""), "ref", wave(2, 1, 1, 0), _route("k_tc_gcnt<3>", "k_tc_tcn2<128>"),
                          True, ("k_tc_gcnt<25,2,128>", "k_tc_tcn2<128>")),
    "gcnt_pairs_wave_over": _c("ntu", (128, 128, 1, True, ""), "ref", wave(2, 1, 1, 1), _route("k_tc_gcnt<3>", "k_tc_tcn2<128>"),
                               True, ("k_tc_gcnt<25,2,128>", "k_tc_tcn2<128>")),
    "tcn2_pairs_wave_over": _c("ntu", (128, 128, 1, True, ""), "ref", wave(2, 2, 1, 1), _route("k_tc_gcnt<3>", "k_tc_tcn2<128>"),
                               True, ("k_tc_gcnt<25,2,128>", "k_tc_tcn2<128>")),
    # token-major graph conv off the tree
    "gcn4_128_offtree_signed": _c("ntu", (128, 128, 1, True, ""), "extra_edge_signed", 7, _route("k_tc_gcn<4>", "k_tc_tcn2<128>"),
                                  True, ("k_tc_gcn<4,2,false>", "k_tc_tcn2<128>")),
    "gcn3_extra_edge": _c("ntu", (128, 256, 2, True, ""), "extra_edge", 7, _route("k_tc_gcn<3>", "k_tc_tcn2<256>"), True,
                          ("k_tc_gcn<3,2,false>", "k_tc_tcn2<256>")),
    "gcnt4_kin_64_128_signed": _c("kinetics", (64, 128, 1, True, ""), "signed", 5, _route("k_tc_gcnt<4>", "k_tc_tcn<128>"), True,
                                  ("k_tc_gcnt<18,1,128>", "k_tc_tcn<128>")),
    "gcn3_256_signed_epi": _c("ntu", (256, 256, 1, True, ""), "signed", 7, _route("k_tc_gcn<3>", "k_tc_tcn2<256>"), True,
                              ("k_tc_gcn<3,2,false>", "k_tc_tcn2<256>")),
    "gcn3_256_nores": _c("ntu", (256, 256, 1, False, ""), "ref", 3, _route("k_tc_gcn<3>", "k_tc_tcn<256>"), True,
                         ("k_tc_gcn<3,2,false>", "k_tc_tcn<256>")),
    "tcn256_pairs_wave_over": _c("kinetics", (256, 256, 1, True, ""), "ref", wave(2, 2, 1, 1), _route("k_tc_gcn<3>", "k_tc_tcn2<256>"),
                                 True, ("k_tc_gcn<3,2,false>", "k_tc_tcn2<256>")),
    # widths the tensor-core kernels were not written for: tensor-core and SIMT kernels hand rings to each other
    "offgrid_32_64": _c("ntu", (32, 64, 1, True, ""), "ref", 7, _route("k_gcn_simt", "k_tcn_simt"), False,
                        ("k_gcn_simt", "k_tcn_simt")),
    "offgrid_64_192": _c("ntu", (64, 192, 1, True, ""), "signed", 7, _route("k_tc_gcn<4>", "k_tcn_simt"), False,
                         ("k_tc_gcn<4,1,false>", "k_tcn_simt")),
    "offgrid_192_192": _c("kinetics", (192, 192, 1, True, ""), "ref", 9, _route("k_tc_gcn<3>", "k_tcn_simt"), False,
                          ("k_tc_gcn<3,2,false>", "k_tcn_simt")),
    "offgrid_96_96": _c("ntu", (96, 96, 1, True, ""), "ref", 7, _route("k_gcn_simt", "k_tcn_simt"), False,
                        ("k_gcn_simt", "k_tcn_simt")),
    "offgrid_simt_gcn_tc_tcn": _c("ntu", (96, 64, 1, False, ""), "ref", 7, _route("k_gcn_simt", "k_tc_tcn<64>"), False,
                                  ("k_gcn_simt", "k_tc_tcn<64>")),
    # first layer: 3 signed input channels (skeleton coordinates in metres)
    "first_layer_small": _c("ntu", (3, 64, 1, False, ""), "ref", 7, _route("k_gcn_small", "k_tc_tcn<64>"), True,
                            ("k_gcn_small", "k_tc_tcn<64>")),
    "first_layer_small_kin": _c("kinetics", (3, 64, 1, False, ""), "signed", 9, _route("k_gcn_small", "k_tc_tcn<64>"), True,
                                ("k_gcn_small", "k_tc_tcn<64>")),
    "plain_8_8_simt": _c("ntu", (8, 8, 1, True, ""), "ref", 7, _route("k_gcn_simt", "k_tcn_simt"), False,
                         ("k_gcn_simt", "k_tcn_simt")),
    # adaptive graph conv
    "agcn_first_small": _c("ntu", (3, 64, 1, False, "adaptive"), "ref", 7, _route("k_attn_small+k_gcn_small", "k_tc_tcn<64>"),
                           False, ("k_attn_small<16,25>", "k_gcn_small", "k_tc_tcn<64>")),
    "agcn_first_small_kin": _c("kinetics", (3, 64, 1, False, "adaptive"), "ref", 9,
                               _route("k_attn_small+k_gcn_small", "k_tc_tcn<64>"), False,
                               ("k_attn_small<16,18>", "k_gcn_small", "k_tc_tcn<64>")),
    "agcn_64_64": _c("ntu", (64, 64, 1, True, "adaptive"), "ref", 7, _route("k_tc_attn+k_tc_agcn", "k_tc_tcn<64>"), False,
                     ("k_tc_attn<16,25>", "k_tc_agcn<4,1,25>", "k_tc_tcn<64>")),
    "agcn_64_64_wave_over": _c("ntu", (64, 64, 1, True, "adaptive"), "ref", wave(1, 1, 1, 1),
                               _route("k_tc_attn+k_tc_agcn", "k_tc_tcn<64>"), False,
                               ("k_tc_attn<16,25>", "k_tc_agcn<4,1,25>", "k_tc_tcn<64>")),
    "agcn_128_128": _c("ntu", (128, 128, 1, True, "adaptive"), "ref", 7, _route("k_tc_attn+k_tc_agcn", "k_tc_tcn2<128>"), False,
                       ("k_tc_attn<32,25>", "k_tc_agcn<3,2,25>", "k_tc_tcn2<128>")),
    "agcn_128_256": _c("ntu", (128, 256, 1, True, "adaptive"), "ref", 7, _route("k_tc_attn+k_tc_agcn", "k_tc_tcn2<256>"), False,
                       ("k_tc_attn<64,25>", "k_tc_agcn<4,1,25>", "k_tc_tcn2<256>")),
    "agcn_kin_64_64": _c("kinetics", (64, 64, 1, True, "adaptive"), "ref", 9, _route("k_tc_attn+k_tc_agcn", "k_tc_tcn<64>"), False,
                         ("k_tc_attn<16,18>", "k_tc_agcn<4,1,18>", "k_tc_tcn<64>")),
    "agcn_kin_64_128": _c("kinetics", (64, 128, 2, True, "adaptive"), "ref", 9, _route("k_tc_attn+k_tc_agcn", "k_tc_tcn2<128>"),
                          False, ("k_tc_attn<32,18>", "k_tc_agcn<4,1,18>", "k_tc_tcn2<128>")),
    "agcn_kin_256_256": _c("kinetics", (256, 256, 1, True, "adaptive"), "ref", 9, _route("k_tc_attn+k_tc_agcn", "k_tc_tcn2<256>"),
                           False, ("k_tc_attn<64,18>", "k_tc_agcn<3,2,18>", "k_tc_tcn2<256>")),
    "agcn_96_simt": _c("ntu", (96, 96, 1, True, "adaptive"), "ref", 7, _route("k_agcn_attn+k_gcn_simt", "k_tcn_simt"), False,
                       ("k_agcn_attn", "k_gcn_simt", "k_tcn_simt")),
    # attention unit (the 64-channel qkv conv is a 128-column single-tap temporal-conv GEMM)
    "sa_64_kin": _c("kinetics", (64, 64, 1, True, "attention"), "ref", 9, _route("k_tc_tcn(qkv)+k_sa_attn", "k_tc_tcn<64>"), False,
                    ("k_sa_affine", "k_tc_tcn2<128>", "k_sa_attn<8>", "k_tc_tcn<64>")),
    "sa_128_kin": _c("kinetics", (128, 128, 1, True, "attention"), "ref", 9, _route("k_tc_sa", "k_tc_tcn2<128>"), False,
                     ("k_sa_affine", "k_tc_sa<16>", "k_tc_tcn2<128>")),
    "sa_128_kin_wave_over": _c("kinetics", (128, 128, 1, True, "attention"), "ref", wave(1, 1, 1, 1),
                               _route("k_tc_sa", "k_tc_tcn2<128>"), False, ("k_sa_affine", "k_tc_sa<16>", "k_tc_tcn2<128>")),
    "sa_64_256_ntu": _c("ntu", (64, 256, 2, True, "attention"), "ref", 7, _route("k_tc_sa", "k_tc_tcn2<256>"), False,
                        ("k_sa_affine", "k_tc_sa<32>", "k_tc_tcn2<256>")),
    "sa_96_128_simt": _c("ntu", (96, 128, 1, True, "attention"), "ref", 7, _route("k_sa_qkv+k_sa_attn", "k_tcn_simt"), False,
                         ("k_sa_qkv", "k_sa_attn<16>", "k_tc_tcn2<128>", "k_tcn_simt")),
    "sa_96_256_simt": _c("ntu", (96, 256, 1, True, "attention"), "ref", 7, _route("k_sa_qkv+k_sa_attn", "k_tcn_simt"), False,
                         ("k_sa_qkv", "k_sa_attn<32>", "k_tc_tcn2<256>", "k_tcn_simt")),
    "sa_96_simt": _c("ntu", (96, 96, 1, True, "attention"), "ref", 7, _route("k_sa_qkv+k_sa_attn", "k_tcn_simt"), False,
                     ("k_sa_qkv", "k_sa_attn_any", "k_tcn_simt")),
}

# test_gpu_routes.py::test_whole_model_signed_input, CoStGcn on NTU among its cases: stepped frame by frame (64 -> 64 blocks as one kernel) and
# time-batched (every block as graph conv + temporal conv), with data_bn, pooling and fc
WHOLE_MODEL_COVERS = ("k_input", "k_gcn_small", "k_tc_tcn<64>", "k_tc_block64", "k_tc_gcn<4,1,false>", "k_tc_gcnt<25,1,128>",
                      "k_tc_gcnt<25,2,128>", "k_tc_gcnt<25,2,256>", "k_tc_tcn<128>", "k_tc_tcn<256>", "k_head")

# Reachable from launch_k but outside the default walks: the k_tc_gcn variants with phase timers (only with COSK_TRACE=1),
# and the unverified k_tc_agcnt (compiled in only with COSK_WITH_AGCNT=1).
EXCLUDED = {f"k_tc_gcn<{p},{s},true>" for p in (3, 4) for s in (1, 2)} | {
    f"k_tc_agcnt<{v},{s},{c}>" for v in (25, 18) for s, c in ((1, 128), (2, 128), (2, 256))}


def covered():
    out = set(WHOLE_MODEL_COVERS)
    for case in ROUTES.values():
        out |= set(case.covers)
    return out


def launched_kernels(path=COSK_CU):
    """Every kernel name passed to launch_k( in cosk.cu; the templated launchers (launch_tc_tcn<COUT> ...) are expanded
    with the template arguments of their call sites."""
    src = re.sub(r"//[^\n]*", "", open(path).read())
    names = set()
    for m in re.finditer(r"launch_k\((k_\w+)(?:<([^>]*)>)?", src):
        name, args = m.group(1), m.group(2)
        if args is None:
            names.add(name)
            continue
        args = [a.strip() for a in args.split(",")]
        if all(re.fullmatch(r"\d+|true|false", a) for a in args):
            names.add(f"{name}<{','.join(args)}>")
            continue
        head = src.rfind("template <", 0, m.start())
        decl = re.match(r"template <([^>]*)>\s*int (\w+)\(", src[head:])
        assert decl, f"no templated launcher around {name}<{args}>"
        params = [p.split()[-1] for p in decl.group(1).split(",")]
        calls = list(re.finditer(rf"\b{decl.group(2)}<([^>]*)>\(", src))
        assert calls, f"{decl.group(2)} is never called"
        for call in calls:
            vals = dict(zip(params, [v.strip() for v in call.group(1).split(",")]))
            names.add(f"{name}<{','.join(vals.get(a, a) for a in args)}>")
    return names
