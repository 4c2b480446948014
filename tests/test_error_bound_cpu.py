"""The per-element error bound of oracle/bound.py, tested on a CPU emulation of the kernels' arithmetic.

The emulator runs one graph conv + temporal conv block the way the tensor-core kernels do: every GEMM operand split
into hi = bf16(a), lo = bf16(a - hi), the products hi*hi + lo*hi + hi*lo summed in fp32, the graph conv as GEMM then
fp32 mix over the vertices, the identity residual as an exact K-block, and every stage result stored as split bf16.
The correct emulation must sit at least 4x inside ``EPS * mag``; each arithmetic fault a kernel could plausibly have
must break the bound on some element (by 4x, except as noted at MUTATIONS).  That is what makes the bound a trustworthy tolerance for the
GPU route tests (tests/test_gpu_routes.py) before any of them runs.

For whole models, ``bound.model`` and ``bound.head`` must compute what the step oracle computes, for all four
architectures, and each plausible fault of the continual head (window length, padding, person mean, rows of two streams
swapped) must break the head's bound by 4x.
"""
import numpy as np
import pytest
import torch

from oracle import bound, regular, step, weights

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


# --- whole models: bound.model and bound.head against the step oracle ---------------------------------------------------
ARCHS = {"cost_gcn": weights.cost_gcn_arch, "cost_gcn_mod": weights.cost_gcn_mod_arch, "coa_gcn": weights.coa_gcn_arch,
         "cos_tr": weights.cos_tr_arch}
# A short window with padding: the first two emissions still hold zero entries, and the window moves on for seven more.
POOL_SIZE, POOL_PADDING, EMISSIONS = 6, 2, 9


def _stepped(tag):
    """Two streams of one model stepped by the oracle in float64: frames, state dict, arch, logits (N, classes, n_emit)
    and the last block's outputs (N*M, C, n, V) in emission order."""
    arch = ARCHS[tag](pool_size=POOL_SIZE, pool_padding=POOL_PADDING)
    sd = weights.make_state_dict(arch, seed=sum(map(ord, tag)), randomize=True)
    first = arch.receptive_field - 1 - arch.stack_padding + (POOL_SIZE - 1 - POOL_PADDING) * arch.stack_stride
    x = weights.make_input((2, 3, first + 1 + (EMISSIONS - 1) * arch.stack_stride, arch.vertices, 2), seed=73).double()
    model = step.StepModel(sd, arch)
    last, seq = model.blocks[-1], []
    last_step = last.step

    def record(h):
        y = last_step(h)
        if y is not None:
            seq.append(y)
        return y

    last.step = record
    with torch.no_grad():
        logits = model.forward_steps(x)
    assert logits.shape[2] == EMISSIONS
    return x, sd, arch, logits, torch.stack(seq, dim=2)


@pytest.fixture(scope="module", params=list(ARCHS))
def stepped(request):
    return (request.param,) + _stepped(request.param)


def _rel(a, b):
    return float((a - b).abs().max()) / float(b.abs().max())


def test_model_oracle_is_the_step_model(stepped):
    tag, x, sd, arch, want, y_seq = stepped
    value, mag = bound.model(x, sd, arch)
    assert value.shape == want.shape
    assert _rel(value, want) <= 1e-12, (tag, _rel(value, want))
    assert bool((mag >= value.abs() - 1e-12).all())


def test_head_oracle_is_the_step_head(stepped):
    tag, x, sd, arch, want, y_seq = stepped
    value, mag = bound.head(y_seq, sd, arch)
    assert value.shape == want.shape
    assert _rel(value, want) <= 1e-12, (tag, _rel(value, want))
    assert bool((mag >= value.abs() - 1e-12).all())


def faulty_head(y, sd, arch, fault):
    """The continual head with one fault, in float64: (N*M, C, n, V) -> (N, classes, n_emit)."""
    P, pp, M = arch.pool_size, arch.pool_padding, arch.persons
    if fault == "rows_swapped":  # stream 0 person 1 and stream 1 person 0: one 128-row token tile holds both
        y = y.clone()
        y[[1, 2]] = y[[2, 1]]
    per_person = y.view(y.shape[0] // M, M, *y.shape[1:]).mean(4)  # (N, M, C, n)
    p = per_person[:, 0] if fault == "one_person" else per_person.mean(1)
    size = {"window_short": P - 1, "window_long": P + 1}.get(fault, P)
    out = []
    for e in range(y.shape[2] - (P - 1 - pp)):
        newest = e + P - 1 - pp
        real = p[:, :, max(0, newest - size + 1): newest + 1]  # entries before input 0 are the window's zeros
        div = real.shape[2] if fault == "padding_dropped" else P
        out.append(torch.nn.functional.linear(real.sum(2) / div, sd["fc.weight"].double(), sd["fc.bias"].double()))
    return torch.stack(out, dim=2)


HEAD_FAULTS = ["window_short", "window_long", "padding_dropped", "one_person", "rows_swapped"]


@pytest.mark.parametrize("fault", HEAD_FAULTS)
def test_each_head_fault_breaks_bound(stepped, fault):
    tag, x, sd, arch, want, y_seq = stepped
    value, mag = bound.head(y_seq, sd, arch)
    assert bound.headroom(faulty_head(y_seq, sd, arch, None), value, mag) <= 1e-6
    h = bound.headroom(faulty_head(y_seq, sd, arch, fault), value, mag)
    print(f"\n[bound] head {tag} {fault}: max err/(EPS*mag) = {h:.3g}")
    assert h >= 4.0, (tag, fault, h)
