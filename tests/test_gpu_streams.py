"""Per-stream state on the GPU (``-m gpu``): reset_streams, export_streams / import_streams and resize_streams on the four
benchmarked workloads at 1037 distinct streams (an odd token-tile count, more tiles than SMs, a ragged last tile).

"Bit-identical" is ``torch.equal`` on emitted logits and on the ``read_block`` rows of every block that emitted.  The
operated-on streams are test_gpu_models._streams' picks: first and last streams, streams whose two skeletons straddle a
token tile, the ragged tile and both sides of the grids' wave boundaries.
"""
import ctypes

import pytest
import torch

import bench
import continual_skeletons_b200 as cs
import test_gpu_models as tgm

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
N = 1037
TAGS = list(tgm.MODELS)


def _model(tag, seed=0, **hp):
    cls, _ = tgm.MODELS[tag]
    bench.set_geometry(tag)
    torch.manual_seed(seed)
    return cls(dict({"dataset_name": bench.DATASET, "forward_mode": "frame"}, **hp))


def _twin(model, tag, **hp):
    other = _model(tag, **hp)
    other.load_state_dict(model.state_dict())
    return other


def _frames(n, seed, count=8):
    gen = torch.Generator().manual_seed(seed)
    return [torch.rand((n, bench.C_IN, bench.V, bench.S), generator=gen).to(DEV) for _ in range(count)]


def _picks(n=N):
    return tgm._streams(n, "kinetics" if bench.V == 18 else "ntu", torch.cuda.get_device_properties(0).multi_processor_count)


def _rows(streams):
    return torch.tensor([2 * n + p for n in streams for p in range(2)], device=DEV)


def _step(model, x):
    out = model.forward_step(x)
    return out, model.last_schedule()


def _same(a_out, a_flags, a, rows_a, b_out, b_flags, b, rows_b, what):
    """Logits and emitted block rows of streams rows_a of model a equal those of rows_b of model b."""
    assert a_flags == b_flags, what
    if a_out is not None:
        sa, sb = rows_a[::2] // 2, rows_b[::2] // 2
        assert torch.equal(a_out[sa], b_out[sb]), what
    for i, fired in enumerate(a_flags[:-1]):
        if fired:
            assert torch.equal(a.read_block(i)[rows_a], b.read_block(i)[rows_b]), (what, i)


def _release(*models):
    for m in models:
        if m._engine is not None:
            m._engine.close()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("tag", TAGS)
def test_reset_leaves_other_streams_alone(tag):
    """B resets the picked streams R at frame F (once mid warm-up, once past it).  For delay + 2 * stride frames every other
    stream -- the skeleton rows sharing a token tile with R included -- is bit-identical to A's.  Every stage has finite
    memory, so once the receptive field has passed after F the reset streams are bit-identical to A's again (the fp64
    pooling sum included: adding and removing the same fp32 values is exact)."""
    a = _model(tag)
    b = _twin(a, tag)
    frames = _frames(N, 1)
    R = _picks()
    others = [n for n in range(N) if n not in set(R)]
    ro, rr = _rows(others), _rows(R)
    sched = a.simulate_schedule(a.delay + 2 * a.stride + 2 + a.receptive_field + a.stride)
    for F in (40, a.delay + 2 * a.stride + 1):
        a.clean_state()
        b.clean_state()
        t = 0
        for t in range(F):
            a.forward_step(frames[t % 8])
            b.forward_step(frames[t % 8])
        b.reset_streams(R)
        back = F + a.receptive_field  # every output from here on was computed from inputs after F only
        for t in range(F, back + a.stride):
            oa, fa = _step(a, frames[t % 8])
            ob, fb = _step(b, frames[t % 8])
            assert fa == sched[t], (tag, t)
            if t < F + a.delay + 2 * a.stride:
                _same(oa, fa, a, ro, ob, fb, b, ro, (tag, F, t, "others"))
            if t >= back:
                _same(oa, fa, a, rr, ob, fb, b, rr, (tag, F, t, "reset streams back"))
    assert a.device_error() == 0 and b.device_error() == 0
    _release(a, b)


@pytest.mark.parametrize("tag", TAGS)
def test_reset_stream_is_a_fresh_stream_on_the_schedule(tag):
    """A stream reset at frame F behaves as a stream whose state was zero at F: resize_streams' fresh streams (zero
    state by construction) and reset streams agree bit for bit."""
    a = _model(tag)
    b = _twin(a, tag)
    frames = _frames(N, 2)
    R = _picks()
    F = a.delay + a.stride + 3
    for t in range(F):
        a.forward_step(frames[t % 8])
        b.forward_step(frames[t % 8])
    a.reset_streams(R)
    b.resize_streams([-1 if n in set(R) else n for n in range(N)])
    rows = _rows(list(range(N)))
    for t in range(F, F + 4 * a.stride):
        oa, fa = _step(a, frames[t % 8])
        ob, fb = _step(b, frames[t % 8])
        _same(oa, fa, a, rows, ob, fb, b, rows, (tag, t))
    _release(a, b)


def _move_case(tag, F, Fc, chunk_a=None):
    """Export the picks of A (N streams) at frame F, import them permuted into C (613 streams, its own history) at frame Fc.
    A steps frame by frame, or through forward_steps in chunks of ``chunk_a`` frames with time_chunk = chunk_a."""
    hp = {"time_chunk": chunk_a} if chunk_a else {}
    a = _model(tag, **hp)
    c = _twin(a, tag, time_chunk=1)
    c0 = _twin(a, tag, time_chunk=1)
    fa, fc = _frames(N, 3), _frames(613, 4)
    picks = _picks()
    gen = torch.Generator().manual_seed(5)
    dest = torch.randperm(613, generator=gen)[: len(picks)].tolist()
    step_a = chunk_a or 1

    def clip(t0, n):
        return torch.stack([fa[t % 8] for t in range(t0, t0 + n)], dim=2)

    for t0 in range(0, F, step_a):
        if chunk_a:
            a.forward_steps(clip(t0, chunk_a))
        else:
            a.forward_step(fa[t0 % 8])
    for t in range(Fc):
        c.forward_step(fc[t % 8])
        c0.forward_step(fc[t % 8])
    st = a.export_streams(picks)
    assert st.meta.frame == F and st.payload.shape == (len(picks), a.stream_bytes())
    c.import_streams(dest, st)
    rp, rd = _rows(picks), _rows(dest)
    keep = [n for n in range(613) if n not in set(dest)]
    rk = _rows(keep)
    pk, dk = torch.tensor(picks, device=DEV), torch.tensor(dest, device=DEV)
    for k in range(0, 4 * a.stride * max(1, step_a // 4) + step_a, step_a):
        xa = clip(F + k, step_a)
        outs_c = []
        for j in range(step_a):
            x = fc[(Fc + k + j) % 8].clone()
            x[dk] = xa[pk, :, j]
            oc, flc = _step(c, x)
            o0, fl0 = _step(c0, fc[(Fc + k + j) % 8])
            _same(oc, flc, c, rk, o0, fl0, c0, rk, (tag, "others", k + j))
            outs_c.append(oc)
        if chunk_a:
            oa = a.forward_steps(xa)
            got = [o for o in outs_c if o is not None]
            if oa is not None:
                oa = oa[..., None] if oa.dim() == 2 else oa
                assert len(got) == oa.shape[-1], (tag, k)
                for e, o in enumerate(got):
                    assert torch.equal(oa[pk, :, e], o[dk]), (tag, k, e)
            for i in range(len(a._specs)):
                assert torch.equal(a.read_block(i)[rp], c.read_block(i)[rd]), (tag, k, i)
        else:
            oa, fla = _step(a, xa[:, :, 0].contiguous())
            _same(oa, fla, a, rp, outs_c[0], c.last_schedule(), c, rd, (tag, "moved", k))
    _release(a, c, c0)


@pytest.mark.parametrize("tag", TAGS)
def test_move_streams_past_warmup(tag):
    a = _model(tag)
    F = a.delay + 2 * a.stride + 1
    _move_case(tag, F, F + 3 * a.stride)


@pytest.mark.parametrize("tag", TAGS)
def test_move_streams_mid_warmup(tag):
    _move_case(tag, 24, 24)


@pytest.mark.parametrize("tag", TAGS)
def test_move_streams_from_a_time_chunked_model(tag, monkeypatch):
    """A steps through forward_steps with time_chunk = 16, C frame by frame.  Stepping and time-batched walks are bit-identical
    with the one-kernel block step off (tests/test_gpu_models.py::test_time_batched_walk_at_scale), so it is off here: what
    is compared is the state that crosses between the two ring sizes."""
    monkeypatch.setenv("COSK_FUSE_BLOCK", "0")
    a = _model(tag)
    F = (a.delay // 16 + 1) * 16
    _move_case(tag, F, F + 2 * a.stride, chunk_a=16)


@pytest.mark.parametrize("tag", TAGS)
def test_roundtrip_is_a_noop_and_swap_moves(tag):
    x = _model(tag)
    y = _twin(x, tag)
    frames = _frames(N, 6)
    F = x.delay + x.stride
    for t in range(F):
        x.forward_step(frames[t % 8])
        y.forward_step(frames[t % 8])
    picks = _picks()
    x.import_streams(picks, x.export_streams(picks))
    allr = _rows(list(range(N)))
    for t in range(F, F + 2 * x.stride):
        ox, fx = _step(x, frames[t % 8])
        oy, fy = _step(y, frames[t % 8])
        _same(ox, fx, x, allr, oy, fy, y, allr, (tag, "roundtrip", t))
    p, q = picks[0], picks[-2]
    x.import_streams([q, p], x.export_streams([p, q]))
    perm = list(range(N))
    perm[p], perm[q] = q, p
    rperm = _rows(perm)
    for t in range(F + 2 * x.stride, F + 4 * x.stride):
        xf = frames[t % 8][torch.tensor(perm, device=DEV)]
        ox, fx = _step(x, xf)
        oy, fy = _step(y, frames[t % 8])
        _same(ox, fx, x, allr, oy, fy, y, rperm, (tag, "swap", t))
    _release(x, y)


@pytest.mark.parametrize("tag", TAGS)
def test_refusals_leave_state_intact(tag):
    a = _model(tag)
    b = _twin(a, tag)
    frames = _frames(N, 7)
    F = a.delay + 2 * a.stride + 1
    for t in range(F):
        a.forward_step(frames[t % 8])
        b.forward_step(frames[t % 8])
    picks = _picks()
    st = a.export_streams(picks)
    with pytest.raises(cs.CoskError):  # a warm-up frame count does not fit a handle past the warm-up
        a.import_streams(picks, cs.StreamState(torch.zeros_like(st.payload), st.meta._replace(frame=10)))
    if a.stride > 1:
        with pytest.raises(cs.CoskError):
            a.import_streams(picks, cs.StreamState(torch.zeros_like(st.payload), st.meta._replace(frame=F + 1)))
    other = "cost_gcn_mod" if tag == "cost_gcn" else "cost_gcn"
    foreign = _model(other)
    foreign.forward_step(_frames(N, 8, 1)[0])
    if foreign.stream_bytes() == a.stream_bytes():
        with pytest.raises(cs.CoskError):
            a.import_streams(picks[:1], foreign.export_streams([0]))
    with pytest.raises(cs.CoskError):
        a.import_streams(picks[:1], cs.StreamState(st.payload[:1], st.meta._replace(geometry=st.meta.geometry ^ 1)))
    for bad in ([N], [-1], [0, 0]):
        for call in (a.reset_streams, a.export_streams):
            with pytest.raises(cs.CoskError):
                call(bad)
        with pytest.raises(cs.CoskError):
            a.import_streams(bad, cs.StreamState(torch.zeros((len(bad), a.stream_bytes()), dtype=torch.uint8, device=DEV), st.meta))
    with pytest.raises(cs.CoskError):
        a.resize_streams([N])
    with pytest.raises(cs.CoskError):  # more streams than 32-bit token rows address: refused after the new geometry is set
        a.resize_streams([-1] * (1 << 22))
    # a handle without state refuses every call
    idx = (ctypes.c_int64 * 1)(0)
    fresh = _model(tag)
    fe = fresh._sync(torch.device(DEV))
    assert fe.lib.cosk_reset_streams(fe.h, idx, 1, None) == -3
    assert fe.lib.cosk_resize_batch(fe.h, 1, idx) == -3
    # a set_batch refused for 32-bit rows leaves the handle's batch as it was (checked before anything is launched on it)
    ae, held = a._engine, a.state_bytes()
    rc = ae.lib.cosk_set_batch(ae.h, 1 << 22)
    assert a.state_bytes() == held
    assert rc == -1
    allr = _rows(list(range(N)))
    for t in range(F, F + 3 * a.stride):
        oa, fa = _step(a, frames[t % 8])
        ob, fb = _step(b, frames[t % 8])
        _same(oa, fa, a, allr, ob, fb, b, allr, (tag, "after refusals", t))
    _release(a, b, foreign, fresh)


@pytest.mark.parametrize("tag", TAGS)
def test_resize_grow_and_shrink(tag):
    """Grow 1037 -> 1100 with fresh streams, then shrink to 500 with a permutation.  Reference: B runs 1100 streams from the
    start (its first 1037 rows on A's inputs) and resets the 63 extra ones at the frame A grows; A's shrunk streams are
    compared with B's rows they came from."""
    a = _model(tag)
    b = _twin(a, tag)
    fa, fx = _frames(N, 9), _frames(1100 - N, 10)
    fb = [torch.cat([x, y]) for x, y in zip(fa, fx)]
    F = a.delay + a.stride + 2
    T = F + 8 * a.stride + 2
    sched = a.simulate_schedule(T)
    for t in range(F):
        a.forward_step(fa[t % 8])
        b.forward_step(fb[t % 8])
    bytes_1037 = a.state_bytes()
    a.resize_streams(list(range(N)) + [-1] * (1100 - N))
    b.reset_streams(list(range(N, 1100)))
    assert a.state_bytes() == b.state_bytes() != bytes_1037
    allr = _rows(list(range(1100)))
    t = F
    for t in range(F, F + 4 * a.stride):
        oa, fla = _step(a, fb[t % 8])
        ob, flb = _step(b, fb[t % 8])
        assert fla == sched[t]
        _same(oa, fla, a, allr, ob, flb, b, allr, (tag, "grown", t))
    gen = torch.Generator().manual_seed(11)
    perm = torch.randperm(1100, generator=gen)[:500].tolist()
    a.resize_streams(perm)
    pk = torch.tensor(perm, device=DEV)
    small = _model(tag)
    small.forward_step(fb[0][:500])
    assert a.state_bytes() == small.state_bytes()
    _release(small)
    for t in range(F + 4 * a.stride, T):
        oa, fla = _step(a, fb[t % 8][pk])
        ob, flb = _step(b, fb[t % 8])
        assert fla == sched[t]
        _same(oa, fla, a, _rows(list(range(500))), ob, flb, b, _rows(perm), (tag, "shrunk", t))
    assert a.device_error() == 0
    _release(a, b)


@pytest.mark.parametrize("tag", TAGS)
def test_each_call_is_one_launch(tag):
    a = _model(tag)
    a.forward_step(_frames(N, 12, 1)[0])
    for idx in ([N // 2], list(range(N))):
        n0 = a.launch_count()
        a.reset_streams(idx)
        assert a.launch_count() == n0 + 1
        st = a.export_streams(idx)
        assert a.launch_count() == n0 + 2
        a.import_streams(idx, st)
        assert a.launch_count() == n0 + 3
    n0 = a.launch_count()
    a.reset_streams([])
    assert a.launch_count() == n0
    _release(a)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_move_between_devices():
    tag = "cost_gcn"
    a = _model(tag)
    c = _twin(a, tag)
    frames = _frames(N, 13)
    F = a.delay + 2 * a.stride + 1
    for t in range(F):
        a.forward_step(frames[t % 8])
        c.forward_step(frames[(t + 3) % 8].to("cuda:1"))
    picks = _picks()
    c.import_streams(picks, a.export_streams(picks))
    rp = _rows(picks)
    for t in range(F, F + 4 * a.stride):
        oa, fa = _step(a, frames[t % 8])
        oc, fc = _step(c, frames[t % 8].to("cuda:1"))
        assert fa == fc
        if oa is not None:
            assert torch.equal(oa[rp[::2] // 2].cpu(), oc[rp[::2].to("cuda:1") // 2].cpu())
        for i, fired in enumerate(fa[:-1]):
            if fired:
                assert torch.equal(a.read_block(i)[rp].cpu(), c.read_block(i)[rp.to("cuda:1")].cpu()), (t, i)
    _release(a, c)
