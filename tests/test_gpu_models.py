"""The four benchmarked models as ``bench.py`` runs them, block by block against the fp64 per-element bound (``-m gpu``).

Each model is built, fed and sized with bench.py's own recipe (its seeds, ``GEOMETRY``/``set_geometry`` and ``SCHED``):
4096 distinct streams, the default pooling windows, stepped with ``forward_step`` past the frame whose logits
``bench.py --dump-outputs`` writes with the default ``--warmup``/``--steps``, and past the wrap of the pooling ring.  On
about 24 streams -- the first and last, both sides of every wave boundary of the one-tile, tile-pair and CTA-pair grids,
streams whose two skeletons sit in different token tiles, and the ragged last tile -- every emitted output of every block
is checked with the single-block bound (``bound.block``, EPS) on the GPU's own emitted output of the block before it,
which is exactly what the kernels consumed: ``read_block`` returns the hi + lo planes of the block-output ring.  The
logits are checked with ``bound.head`` on the GPU's last-block outputs, and end to end with ``bound.model`` (the bound
chained through the stack, n_blocks * EPS).

A negative control scales one output channel of one temporal conv by 1 + 2^-8 in the GPU model only: the check must
flag that block and no other.  The time-batched walk is run at 4096 streams with a time chunk whose 256-channel ring
holds more than 2^31 elements.

Printed per model: max |got - value| / (EPS * mag) per block and for the logits, and the GPU and CPU-oracle seconds.
"""
import gc
import time

import pytest
import torch

import bench
import continual_skeletons_b200 as cs
import route_table
from oracle import bound, weights

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
MODELS = {
    # tag: (class, oracle arch factory)
    "cost_gcn": (cs.CoStGcn, weights.cost_gcn_arch),
    "cost_gcn_mod": (cs.CoStGcnMod, weights.cost_gcn_mod_arch),
    "coa_gcn": (cs.CoAGcn, weights.coa_gcn_arch),
    "cos_tr": (cs.CoSTr, weights.cos_tr_arch),
}
N_STREAMS = 4096
BENCH_WARMUP, BENCH_STEPS = 8, 200  # bench.py's default --warmup / --steps
ROWS_PER_ORACLE_CALL = 16  # skeletons per bound.block call: bounds the oracle's memory on the longest sequences


def _oracle_state(model):
    """A copy of the model's own parameters under the regular key names (the inverse of map_state_dict's key
    shortening)."""
    return {k.replace("0.1.", "").replace("0.0.residual", "residual"): v.detach().cpu().clone()
            for k, v in model.state_dict().items()}


def _build(tag, n_streams, **hp):
    """bench.py's model and input frames for ``tag``: (model, oracle state dict, oracle arch, the 8 cycled frames)."""
    cls, arch_fn = MODELS[tag]
    bench.set_geometry(tag)
    skel = "kinetics" if bench.V == 18 else "ntu"
    torch.manual_seed(0)
    model = cls(dict({"dataset_name": bench.DATASET, "forward_mode": "frame"}, **hp))
    sd = _oracle_state(model)
    arch = arch_fn(skeleton=skel, classes=bench.CLASSES)
    assert arch.vertices == bench.V and (arch.pool_size, arch.pool_padding) == (model.pool_size, model.pool_padding)
    gen = torch.Generator().manual_seed(1234)
    frames = [torch.rand((n_streams, bench.C_IN, bench.V, bench.S), generator=gen) for _ in range(8)]
    return model, sd, arch, frames


def _streams(n_streams, skel, sms):
    """The checked streams: both sides of the grids' wave boundaries (route_table.picked, in skeletons), the first and
    last, three streams whose two skeletons straddle a token-tile boundary, and the ragged last tile and the one before."""
    spt = route_table.SPT[skel]
    pick = {s // 2 for s in route_table.picked(2 * n_streams, skel, sms)}
    straddle = [n for n in range(n_streams) if (2 * n + 1) % spt == 0]
    pick |= {straddle[0], straddle[len(straddle) // 2], straddle[-1]}
    last_tile = (2 * n_streams - 1) // spt * spt  # first skeleton of the last (ragged) tile
    pick |= {last_tile // 2, last_tile // 2 - 1, n_streams - 1}
    return sorted(pick)


def _clip(frames, streams, n):
    """The first ``n`` cycled frames of ``streams``: (len(streams), C, n, V, S)."""
    return torch.stack([frames[t % 8][streams] for t in range(n)], dim=2)


def _block(x, sd, name, spec, pad, xm):
    """bound.block over groups of skeletons."""
    outs = [bound.block(x[r: r + ROWS_PER_ORACLE_CALL], sd, name, spec, pad,
                        xm=None if xm is None else xm[r: r + ROWS_PER_ORACLE_CALL])
            for r in range(0, x.shape[0], ROWS_PER_ORACLE_CALL)]
    return torch.cat([o[0] for o in outs]), torch.cat([o[1] for o in outs])


def check_blocks(x, sd, arch, seqs):
    """Headroom of every block: block 0 on the data_bn-normalised frames ``x`` (N, C, T, V, S), block i on ``seqs[i-1]``,
    the GPU's emitted outputs of block i - 1 (N*S, C, n, V).  Returns max err / (EPS * mag) per block."""
    h, hm = bound.data_bn(x, sd)
    out = []
    for name, spec, got in zip(arch.block_names, arch.blocks, seqs):
        value, mag = _block(h, sd, name, spec, arch.padding, hm)
        n = got.shape[2]
        assert value.shape[2] >= n, (name, value.shape, got.shape)
        out.append(bound.headroom(got, value[:, :, :n], mag[:, :, :n]))
        h, hm = got.double(), None
    return out


def run_stepped(model, frames, n_frames, streams):
    """Steps ``model`` over ``n_frames`` cycled frames and keeps, of the picked streams, every emitted output of every block
    (N*S, C, n_i, V) and the logits (N, classes, n_emit).  The emission flags must match simulate_schedule every frame."""
    rows = torch.tensor([2 * n + p for n in streams for p in range(2)], device=DEV)
    cols = torch.tensor(streams, device=DEV)
    dev_frames = [f.to(DEV) for f in frames]
    sched = model.simulate_schedule(n_frames)
    n_blocks = len(sched[0]) - 1
    seqs, logits = [[] for _ in range(n_blocks)], []
    for t in range(n_frames):
        out = model.forward_step(dev_frames[t % 8])
        flags = model.last_schedule()
        assert flags == sched[t], (t, flags, sched[t])
        for i in range(n_blocks):
            if flags[i]:
                seqs[i].append(model.read_block(i)[rows].cpu())
        if out is not None:
            logits.append(out[cols].cpu())
    assert model.device_error() == 0, hex(model.device_error())
    seqs = [torch.stack(s, dim=2) for s in seqs]
    return seqs, (torch.stack(logits, dim=2) if logits else None)


def _release(model):
    model._engine.close()
    del model
    gc.collect()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("tag", list(MODELS))
def test_bench_model_block_by_block(tag):
    model, sd, arch, frames = _build(tag, N_STREAMS)
    warm, period = bench.SCHED[tag]
    # the timed steps of bench.py end at frame warm + warmup + steps; the pooling ring wraps pool_size emissions in
    n_frames = max(warm + BENCH_WARMUP + BENCH_STEPS, warm + (arch.pool_size + 1) * period) + 1
    streams = _streams(N_STREAMS, arch.skeleton, torch.cuda.get_device_properties(0).multi_processor_count)
    t0 = time.perf_counter()
    seqs, logits = run_stepped(model, frames, n_frames, streams)
    gpu_s = time.perf_counter() - t0
    _release(model)
    t0 = time.perf_counter()
    x = _clip(frames, streams, n_frames)
    with torch.no_grad():
        heads = check_blocks(x, sd, arch, seqs)
        value, mag = bound.head(seqs[-1], sd, arch)
        assert logits is not None and logits.shape == value.shape, (None if logits is None else logits.shape, value.shape)
        h_head = bound.headroom(logits, value, mag)
        value, mag = bound.model(x, sd, arch)
        assert logits.shape == value.shape
        h_model = bound.headroom(logits, value, len(arch.blocks) * mag)
    cpu_s = time.perf_counter() - t0
    print(f"\n[models] {tag} {N_STREAMS} streams, {len(streams)} checked, {n_frames} frames, {logits.shape[2]} emissions: "
          f"headroom per block " + " ".join(f"{h:.3f}" for h in heads) +
          f" | head {h_head:.3f} | model (10 EPS) {h_model:.3f} | GPU {gpu_s:.1f} s, CPU oracle {cpu_s:.1f} s")
    assert max(heads) <= 1.0, (tag, heads)
    assert h_head <= 1.0, (tag, h_head)
    assert h_model <= 1.0, (tag, h_model)


def test_perturbed_temporal_conv_is_flagged_at_its_block_only():
    """Layer 8 (block index 7) has one output channel of its temporal conv scaled by 1 + 2^-8 in the GPU model only.  Its
    outputs break the bound; blocks 8 and 9, which consume them, and every earlier block still pass.

    A fault in a channel that the ReLU zeroes everywhere would be invisible, so the perturbed channel is the one the
    ReLU lets through most often in an unperturbed run."""
    n_streams, perturbed = 12, 7
    model, sd, arch, frames = _build("cost_gcn", n_streams)
    n_frames = arch.receptive_field + 4 * arch.stack_stride  # block 9 emits five times
    streams = list(range(n_streams))
    seqs, _ = run_stepped(model, frames, n_frames, streams)
    channel = int((seqs[perturbed] > 0).sum(dim=(0, 2, 3)).argmax())
    with torch.no_grad():
        model.get_parameter("layers.layer8.0.1.tcn.t_conv.weight")[channel] *= 1.0 + 2.0 ** -8
    model.sync_weights()  # re-uploads the weights; the next step starts from a fresh state
    seqs, _ = run_stepped(model, frames, n_frames, streams)
    _release(model)
    with torch.no_grad():
        heads = check_blocks(_clip(frames, streams, n_frames), sd, arch, seqs)
    print(f"\n[models] cost_gcn, layer 8 channel {channel} perturbed: headroom per block " + " ".join(f"{h:.3f}" for h in heads))
    assert heads[perturbed] > 1.0, heads
    assert all(h <= 1.0 for i, h in enumerate(heads) if i != perturbed), heads


def ring_elements(n_streams, V, persons, cout, time_chunk):
    """Elements of one temporal ring as cosk_set_batch_ex allocates it: (8 + time_chunk) slots of hi and lo planes of
    t_alloc token rows."""
    spt = 128 // V
    n_tiles = -(-n_streams * persons // spt)
    t_alloc = ((n_tiles + 1) * spt * V + (128 - spt * V) + 7) // 8 * 8
    return (8 + time_chunk) * 2 * t_alloc * cout


@pytest.mark.parametrize("tag", ["cost_gcn", "cost_gcn_mod"])
def test_time_batched_walk_at_scale(tag, monkeypatch):
    """forward_steps over 4096 distinct streams with the automatic time chunk and with 16 frames per chunk, where one
    256-channel ring holds more than 2^31 elements.  With the one-kernel block step off both equal stepping frame by
    frame bit for bit; with the default kernels both hold to bound.model on the checked streams."""
    big = 16
    bench.set_geometry(tag)
    assert ring_elements(N_STREAMS, bench.V, bench.S, 256, big) > 2 ** 31
    warm, period = bench.SCHED[tag]
    n_frames = warm + 2 * period  # three emissions: the warm frames end with the first

    def run(tc, stepped=False):
        model, sd, arch, frames = _build(tag, N_STREAMS, time_chunk=tc)
        x = _clip(frames, list(range(N_STREAMS)), n_frames).to(DEV)
        if stepped:
            outs = [model.forward_step(x[:, :, t].contiguous()) for t in range(n_frames)]
            got = torch.stack([o for o in outs if o is not None], dim=2)
        else:
            got = model.forward_steps(x)
            assert model._engine.time_chunk == tc if tc > 0 else model._engine.time_chunk > 1, model._engine.time_chunk
        assert model.device_error() == 0, hex(model.device_error())
        _release(model)
        del x
        return got.cpu(), sd, arch, frames

    monkeypatch.setenv("COSK_FUSE_BLOCK", "0")
    want = run(1, stepped=True)[0]
    assert want.shape == (N_STREAMS, 60, 3)
    for tc in (-1, big):
        assert torch.equal(run(tc)[0], want), tc
    monkeypatch.delenv("COSK_FUSE_BLOCK")
    for tc in (-1, big):
        got, sd, arch, frames = run(tc)
        streams = _streams(N_STREAMS, arch.skeleton, torch.cuda.get_device_properties(0).multi_processor_count)
        with torch.no_grad():
            value, mag = bound.model(_clip(frames, streams, n_frames), sd, arch)
        h = bound.headroom(got[streams], value, len(arch.blocks) * mag)
        print(f"\n[models] {tag} forward_steps time_chunk={tc}: logits max err/(10*EPS*mag) = {h:.3f}")
        assert h <= 1.0, (tag, tc, h)
