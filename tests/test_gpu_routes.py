"""Route matrix (``-m gpu``): one block per case, chosen so that the dispatcher in csrc/cosk.cu takes a given kernel
route, checked element by element against the fp64 oracle with the per-element bound of oracle/bound.py.

Each case names the adjacency it loads (through ``gcn.A`` / ``gcn.graph_attn``), the block shape, the skeleton and the
skeleton count, and the kernels ``knobs()`` must report for it.  Every case then runs three walks -- ``forward_step``
frame by frame, ``forward_steps`` with the automatic time chunk, and ``forward_steps(pad_end=True)`` with a chunk that
wraps the rings -- and checks

* the route: the kernel names of ``knobs()["blocks"][0]``;
* ``device_error() == 0``;
* ``|got - value| <= EPS * mag`` on every emitted frame and element of the checked streams (all of them, or at large
  counts the first and last streams and those on both sides of every wave boundary of the grid);
* ``forward_steps`` with ``time_chunk=1`` == ``forward_step`` bit for bit, and frame-by-frame == time-batched bit for bit
  where both run the same kernels.  The one-kernel 64 -> 64 block step (k_tc_block64) is only compared within the
  bound: time-batched chunks run such a block as graph conv + temporal conv launches, which round differently.
* a stack time-batched chunks cannot take falls back to stepping (same launch count as stepping).

The table, with the kernels each case launches, lives in tests/route_table.py; tests/test_boundary_cpu.py checks that
it declares every kernel csrc/cosk.cu can launch.  test_whole_model_signed_input runs the first-layer path with data_bn
and the head (k_input, k_gcn_small, k_head) on signed skeleton coordinates through each of the four whole models, on
both skeletons.

The printed figure per case is max |got - value| / (EPS * mag), the headroom observed on the GPU.
"""
import numpy as np
import pytest
import torch

import continual_skeletons_b200 as cs
import route_table
from oracle import bound, weights
from route_table import ROUTES

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
T = 12  # frames per clip: the first emission is at frame 4 (padding 4), the ring of 9 taps wraps


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _state(tag):
    case = ROUTES[tag]
    cin, cout, stride, residual, gconv = case.shape
    spec = weights.BlockSpec(cin, cout, stride, residual, gconv)
    arch = weights.ArchSpec([spec], padding=4, skeleton=case.skel, head=False, block_names=["0."],
                            graph_conv="adaptive" if gconv == "adaptive" else "plain")
    seed = sum(map(ord, tag))
    sd = weights.make_state_dict(arch, seed=seed, randomize=True)
    rng = np.random.Generator(np.random.PCG64(seed + 1))
    if gconv != "attention":
        A, ga = route_table.adjacency(case.adj, case.skel, rng)
        if gconv == "adaptive":
            ga = ga * 0.05 if case.adj == "ref" else ga
        sd["0.gcn.A"], sd["0.gcn.graph_attn"] = A, ga
    kind = spec.res_kind
    mapped = {}
    for k, v in sd.items():
        rest = k.split(".", 1)[1]
        mapped[f"0.{rest}" if kind == 0 else (f"0.0.0.{rest}" if rest.startswith("residual") else f"0.0.1.{rest}")] = v
    B = route_table.skeletons(case.n, case.skel, _sms())
    V = arch.vertices
    if cin == 3:
        x = route_table.signed_coordinates(rng, (B, 3, T, V), case.skel)
    else:
        x = torch.from_numpy(rng.uniform(-1.0, 1.0, size=(B, cin, T, V)).astype(np.float32))
    return spec, sd, mapped, x


def _stack(tag, mapped, tc):
    case = ROUTES[tag]
    st = cs.CoStack([cs.BlockSpec(*case.shape)], padding=4, skeleton=case.skel, kernel_path=case.path, time_chunk=tc)
    st.load_state_dict(mapped, strict=True)
    return st


def _check_route(st, want):
    got = st.knobs()["blocks"][0]
    if "block" in want:
        assert "block" in got and got["block"].startswith(want["block"]), got
    else:
        assert "block" not in got, got
        assert got["gcn"].startswith(want["gcn"]), got
        assert got["tcn"] == want["tcn"], got


@pytest.mark.parametrize("tag", list(ROUTES))
def test_route(tag):
    case = ROUTES[tag]
    spec, sd, mapped, x = _state(tag)
    B = x.shape[0]
    pick = route_table.picked(B, case.skel, _sms())
    value, mag = bound.block(x[pick].double(), sd, "0.", spec, 4)
    xd = x.to(DEV)
    # frame by frame
    st = _stack(tag, mapped, 1)
    outs = []
    for t in range(T):
        o = st.forward_step(xd[:, :, t].contiguous())
        if t == 0:
            _check_route(st, case.route)
        if o is not None:
            outs.append(o)
    assert st.device_error() == 0, hex(st.device_error())
    stepped = torch.stack(outs, dim=2)
    step_launches = st.launch_count()
    n = stepped.shape[2]
    h_step = bound.headroom(stepped[pick].cpu(), value[:, :, :n], mag[:, :, :n])
    # forward_steps one frame per chunk: the same kernels as stepping
    st1 = _stack(tag, mapped, 1)
    one = st1.forward_steps(xd)
    assert st1.device_error() == 0, hex(st1.device_error())
    assert st1.launch_count() == step_launches, (st1.launch_count(), step_launches)
    assert torch.equal(one, stepped)
    # whole clip in one time-batched call (or stepped inside the library when the stack is not eligible)
    st2 = _stack(tag, mapped, -1)
    whole = st2.forward_steps(xd)
    assert st2.device_error() == 0, hex(st2.device_error())
    _check_route(st2, case.route)
    if case.batched:
        assert st2.launch_count() < step_launches, (st2.launch_count(), step_launches)
    else:
        assert st2.launch_count() == step_launches, (st2.launch_count(), step_launches)
    if "block" not in case.route:
        assert torch.equal(whole, stepped)
    h_whole = bound.headroom(whole[pick].cpu(), value[:, :, :n], mag[:, :, :n])
    # the full clip with the end padding flushed, in chunks of 5 frames (the rings wrap inside a chunk)
    st3 = _stack(tag, mapped, 5)
    full = st3.forward_steps(xd, pad_end=True)
    assert st3.device_error() == 0, hex(st3.device_error())
    assert full.shape[2] == value.shape[2], (full.shape, value.shape)
    h_full = bound.headroom(full[pick].cpu(), value, mag)
    h = max(h_step, h_whole, h_full)
    print(f"\n[route] {tag}: B={B} checked={len(pick)} knobs={st.knobs()['blocks'][0]} "
          f"max err/(EPS*mag) step={h_step:.4f} steps={h_whole:.4f} pad_end={h_full:.4f}")
    assert h <= 1.0, (tag, h_step, h_whole, h_full)


WHOLE_MODELS = {"cost_gcn": (cs.CoStGcn, weights.cost_gcn_arch), "cost_gcn_mod": (cs.CoStGcnMod, weights.cost_gcn_mod_arch),
                "coa_gcn": (cs.CoAGcn, weights.coa_gcn_arch), "cos_tr": (cs.CoSTr, weights.cos_tr_arch)}


@pytest.mark.parametrize("skel", ["ntu", "kinetics"])
@pytest.mark.parametrize("tag", list(WHOLE_MODELS))
def test_whole_model_signed_input(tag, skel):
    """A whole model on signed skeleton coordinates (data_bn folded into k_input, the first layer's graph conv, ten blocks,
    pooling and fc in k_head), stepped frame by frame and time-batched, against ``bound.model``: the model in float64
    with the block bound chained through the stack, which holds the logits to n_blocks * EPS * mag.  The window has two
    entries of padding, so the first emissions average over its zeros."""
    cls, arch_fn = WHOLE_MODELS[tag]
    classes = 60 if skel == "ntu" else 400
    P, pp = 8, 2
    arch = arch_fn(skeleton=skel, classes=classes, pool_size=P, pool_padding=pp)
    sd = weights.make_state_dict(arch, seed=91, randomize=True)
    first = arch.receptive_field - 1 - arch.stack_padding + (P - 1 - pp) * arch.stack_stride
    Tm = first + 1 + 2 * arch.stack_stride  # three emissions
    rng = np.random.Generator(np.random.PCG64(92))
    x = route_table.signed_coordinates(rng, (2, 3, Tm, arch.vertices, 2), skel)
    with torch.no_grad():
        want, mag = bound.model(x, sd, arch)  # (N, classes, 3)
    tol = len(arch.blocks) * bound.EPS
    for tc in (1, -1):
        model = cls({"dataset_name": "dummy_ntu" if skel == "ntu" else "dummy_kin", "pool_size": P, "pool_padding": pp,
                     "time_chunk": tc})
        model.load_state_dict(model.map_state_dict(sd), strict=True)
        got = model.forward_steps(x.to(DEV))
        assert model.device_error() == 0, hex(model.device_error())
        assert tuple(got.shape) == tuple(want.shape), (got.shape, want.shape)
        r = float(((got.cpu().double() - want).abs() / (tol * mag + bound.TINY)).max())
        print(f"\n[route] whole {tag} {skel} time_chunk={tc}: knobs={model.knobs()['blocks'][:2]} "
              f"max err/({len(arch.blocks)}*EPS*mag) = {r:.4f}")
        assert r <= 1.0, (tag, skel, tc, r)
