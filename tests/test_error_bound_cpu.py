"""The per-element error bound of oracle/bound.py, tested on a CPU emulation of the kernels' arithmetic.

The emulator runs one graph conv + temporal conv block the way the tensor-core kernels do: every GEMM operand split
into hi = bf16(a), lo = bf16(a - hi), the products hi*hi + lo*hi + hi*lo summed in fp32, the graph conv as GEMM then
fp32 mix over the vertices, the identity residual as an exact K-block, and every stage result stored as split bf16.
The correct emulation must sit at least 4x inside ``EPS * mag``; each arithmetic fault a kernel could plausibly have
must break the bound on some element (by 4x, except as noted at MUTATIONS).  That is what makes the bound a trustworthy tolerance for the
GPU route tests (tests/test_gpu_routes.py) before any of them runs.
"""
import numpy as np
import pytest
import torch

from oracle import bound, regular, weights

SKEL_PER_TILE = {"ntu": 5, "kinetics": 7}  # 128 token rows per tile / V


def split(a):
    hi = a.to(torch.bfloat16).float()
    return hi, (a - hi).to(torch.bfloat16).float()


def mm(x, w, drop_hilo=False, w_lo_zero_cols=None):
    """x (N, K) fp32 @ w (M, K)^T in split-bf16 products with fp32 sums."""
    xh, xl = split(x)
    wh, wl = split(w)
    if w_lo_zero_cols is not None:
        wl = wl.clone()
        wl[:, w_lo_zero_cols] = 0
    y = xh @ wh.T + xl @ wh.T
    if not drop_hilo:
        y = y + xh @ wl.T
    return y


def store(y, without_lo=False):
    hi, lo = split(y)
    return hi if without_lo else hi + lo


def fold(sd, conv, bn):
    w, b, _ = bound._folded(sd, conv, bn)
    return w[:, :, :, 0].float(), b.float()


def emulate(x, sd, key, spec, pad, skel, mut=()):
    """x (B, Cin, T, V) -> block output (B, Cout, T_out, V) in fp32, the kernels' arithmetic.  ``mut``: faults."""
    B, C, T, V = x.shape
    g = key + "gcn."
    s = bound._folded(sd, g + "g_conv.0.", g + "bn.")[2]
    Wp = [(sd[g + f"g_conv.{p}.weight"].double()[:, :, 0, 0] * s[:, None]).float() for p in range(3)]
    bias = (s * sum(sd[g + f"g_conv.{p}.bias"].double() for p in range(3)) + sd[g + "bn.bias"].double()
            - sd[g + "bn.running_mean"].double() * s)
    mix = (sd[g + "A"].double() * sd[g + "graph_attn"].double()).float().clone()
    if "mix_bf16" in mut:  # mixing coefficients kept in bf16 only: each off by up to 2^-9 relative
        mix = mix.to(torch.bfloat16).float()
    xin = store(x.float().permute(0, 2, 3, 1).reshape(-1, C))  # tokens (B, T, V) x C, split on input
    res = 0
    if (g + "gcn_residual.0.weight") in sd:
        Wr, br = fold(sd, g + "gcn_residual.0.", g + "gcn_residual.1.")
        res = mm(xin, Wr[:, :, 0])
        bias = bias + br.double()
    else:
        res = xin
    cout = Wp[0].shape[0]
    y = 0
    for p in range(3):
        yp = mm(xin, Wp[p], drop_hilo="drop_hilo" in mut).reshape(B * T, V, cout)
        y = y + torch.einsum("vw,nvc->nwc", mix[p], yp)
    y = torch.relu(y.reshape(-1, cout) + res + bias.float())
    G = store(y, without_lo="store_without_lo" in mut).reshape(B, T, V, cout)
    # temporal conv: 9 taps (+ residual K-block) as one GEMM
    st = spec.stride
    Gp = torch.nn.functional.pad(G, (0, 0, 0, 0, pad, pad))
    T_out = (T + 2 * pad - 9) // st + 1
    taps = torch.stack([Gp[:, k: k + st * (T_out - 1) + 1: st] for k in range(9)], dim=3)  # (B, T_out, V, 9, C)
    A = taps.reshape(-1, 9 * cout)
    Wt, bt = fold(sd, key + "tcn.t_conv.", key + "tcn.bn.")
    Wt = Wt.permute(0, 2, 1).reshape(cout, 9 * cout)
    shrink = 4 - pad
    xs = x.float()[:, :, shrink: T - shrink] if shrink else x.float()
    xs = store(xs[:, :, ::st][:, :, :T_out].permute(0, 2, 3, 1).reshape(-1, C))
    if spec.res_kind == 1:
        A, Wt = torch.cat([A, xs], 1), torch.cat([Wt, torch.eye(cout)], 1)
    elif spec.res_kind == 2:
        Wr, br = fold(sd, key + "residual.t_conv.", key + "residual.bn.")
        A, Wt, bt = torch.cat([A, xs], 1), torch.cat([Wt, Wr[:, :, 0]], 1), bt + br
    cols = list(range(4 * cout, 5 * cout)) if "tap_bf16" in mut else None
    out = torch.relu(mm(A, Wt, drop_hilo="drop_hilo" in mut, w_lo_zero_cols=cols) + bt)
    out = store(out, without_lo="store_without_lo" in mut).reshape(B, T_out, V, cout).permute(0, 3, 1, 2).contiguous()
    if "stale_last_token" in mut:  # the last token of the ragged last tile never written
        assert B % SKEL_PER_TILE[skel] != 0
        out[B - 1, :, :, V - 1] = 0
    return out


CASES = {
    # tag: (skeleton, BlockSpec, skeletons, frames)
    "ntu_64_64_identity": ("ntu", weights.BlockSpec(64, 64, 1, True), 7, 14),
    "kinetics_128_128_identity": ("kinetics", weights.BlockSpec(128, 128, 1, True), 9, 14),
}
# fault -> least max err / (EPS * mag) it must reach.  Coefficients rounded to bf16 move each mixed term by <= 2^-9,
# diluted over the three partitions, the taps and the residual: caught, but with less than 4x to spare.
MUTATIONS = {"drop_hilo": 4.0, "store_without_lo": 4.0, "tap_bf16": 4.0, "mix_bf16": 1.5, "stale_last_token": 4.0}


def _setup(tag):
    skel, spec, B, T = CASES[tag]
    arch = weights.ArchSpec([spec], padding=4, skeleton=skel, head=False, block_names=["b."])
    sd = weights.make_state_dict(arch, seed=71, randomize=True)
    rng = np.random.Generator(np.random.PCG64(72))
    # signed coefficients: four-part weights, no cancellation-free sums
    sd["b.gcn.graph_attn"] = torch.from_numpy(rng.uniform(-1.5, 1.5, size=tuple(sd["b.gcn.graph_attn"].shape)).astype(np.float32))
    x = torch.from_numpy(rng.uniform(-2.0, 4.0, size=(B, spec.cin, T, arch.vertices)))
    value, mag = bound.block(x, sd, "b.", spec, 4)
    return skel, spec, sd, x, value, mag


@pytest.fixture(scope="module", params=list(CASES))
def case(request):
    return (request.param,) + _setup(request.param)


def test_oracle_value_is_the_regular_block(case):
    tag, skel, spec, sd, x, value, mag = case
    assert torch.equal(value, regular.st_block(x.double(), sd, "b.", spec, 4))
    assert bool((mag >= value.abs() - 1e-12).all())


def test_correct_emulation_within_quarter_of_bound(case):
    tag, skel, spec, sd, x, value, mag = case
    got = emulate(x, sd, "b.", spec, 4, skel)
    assert got.shape == value.shape
    h = bound.headroom(got, value, mag)
    print(f"\n[bound] {tag} correct: max err/(EPS*mag) = {h:.4f}")
    assert h <= 0.25, h


@pytest.mark.parametrize("mut", list(MUTATIONS))
def test_each_fault_breaks_bound(case, mut):
    tag, skel, spec, sd, x, value, mag = case
    got = emulate(x, sd, "b.", spec, 4, skel, mut=(mut,))
    h = bound.headroom(got, value, mag)
    print(f"\n[bound] {tag} {mut}: max err/(EPS*mag) = {h:.2f}")
    assert h >= MUTATIONS[mut], (mut, h)
