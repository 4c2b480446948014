"""prime_streams on the GPU (``-m gpu``): joining streams primed from their recent frames, on the four benchmarked workloads
at 1037 distinct streams (helpers of test_gpu_streams / test_gpu_models; the primed streams are test_gpu_streams._picks).

A and B are twin handles.  In A the picked streams are reset at F - H' (H' = min(H, F)) and then receive their clip
frames while the other streams receive their own; in B the picked streams receive different frames until F and are
primed there from the clip.  After the call the payloads of all N streams are bit-identical between A and B, and so are
the logits and the ``read_block`` rows of every emission for the next ``receptive_field + stride`` frames.  Where the
walks being compared differ in time chunk, the one-kernel block step is off (COSK_FUSE_BLOCK=0), which makes stepping
and time-batched walks bit-identical (tests/test_gpu_models.py::test_time_batched_walk_at_scale).
"""
import ctypes

import pytest
import torch

import bench
import continual_skeletons_b200 as cs
import test_gpu_models as tgm
import test_gpu_streams as tgs
from oracle import bound

pytestmark = pytest.mark.gpu

DEV = tgs.DEV
N = tgs.N
TAGS = tgs.TAGS
ORACLE_STREAMS = 4  # picked streams checked against bound.model (the fp64 oracle's cost grows with streams x frames)


def _cases(m, mode):
    """(F, H) pairs: H' below the warm-up, H' = receptive_field, H > F (clipped, past the warm-up), H = 0, H not a multiple
    of the stride, F at every phase modulo the stride."""
    rf, s, warm = m.receptive_field, m.stride, m.delay
    if mode == "chunk1":
        return [(61, 37), (rf + 2, rf), (warm + 10, warm + 17), (30, 0)]
    if mode == "auto":
        return [(100 + p, 45 + p) for p in range(s)] + [(rf + 3, rf + 1)]
    return [(rf + 5, rf + 8)]  # tc16


def _history(picks, seed):
    """The picked streams' own frames, 8 cycled frames of (len(picks), C, V, S)."""
    return tgs._frames(len(picks), seed)


def _feed(x, pk, y, t):
    x = x.clone()
    x[pk] = y[t % 8]
    return x


def _export_all(m):
    return m.export_streams(list(range(N))).payload


@pytest.mark.parametrize("mode", ["chunk1", "auto", "tc16"])
@pytest.mark.parametrize("tag", TAGS)
def test_primed_equals_reset_and_fed(tag, mode, monkeypatch):
    """chunk1: default kernels, main handles and priming walk frame by frame (time_chunk = 1).  auto: main handles step
    frame by frame, priming picks its chunk (_pick_time_chunk).  tc16: main handles hold rings for 16-frame chunks and
    priming walks 16-frame chunks."""
    if mode != "chunk1":
        monkeypatch.setenv("COSK_FUSE_BLOCK", "0")
    hp = {"chunk1": {"time_chunk": 1}, "auto": {}, "tc16": {"time_chunk": 16}}[mode]
    a = tgs._model(tag, **hp)
    b = tgs._twin(a, tag, **hp)
    xs = tgs._frames(N, 21)
    picks = tgs._picks()
    pk = torch.tensor(picks, device=DEV)
    others = [n for n in range(N) if n not in set(picks)]
    ys, zs = _history(picks, 22), _history(picks, 23)  # the picks' clip frames; B's picks' frames before priming
    allr = tgs._rows(list(range(N)))
    for F, H in _cases(a, mode):
        Hp = min(H, F)
        a.clean_state()
        b.clean_state()
        for t in range(F):
            if 0 < t == F - Hp:  # at t = 0 the state is zero already
                a.reset_streams(picks)
            a.forward_step(_feed(xs[t % 8], pk, ys, t) if t >= F - Hp else xs[t % 8])
            b.forward_step(_feed(xs[t % 8], pk, zs, t))
        if Hp == 0:
            a.reset_streams(picks)
        clip = torch.stack([ys[t % 8] for t in range(F - H, F)], dim=2) if H else \
            torch.empty((len(picks), bench.C_IN, 0, bench.V, bench.S), device=DEV)
        before, flags_before = _export_all(b), b.last_schedule()
        b.prime_streams(picks, clip)
        after = _export_all(b)
        assert b.frame_count() == F and b.last_schedule() == flags_before, (tag, mode, F, H)
        assert torch.equal(after[others], before[others]), (tag, mode, F, H, "others")
        assert torch.equal(after, _export_all(a)), (tag, mode, F, H, "primed")
        sched = a.simulate_schedule(F + a.receptive_field + a.stride)
        for t in range(F, F + a.receptive_field + a.stride):
            x = _feed(xs[t % 8], pk, ys, t)
            oa, fa = tgs._step(a, x)
            ob, fb = tgs._step(b, x)
            assert fb == sched[t], (tag, mode, F, H, t)
            tgs._same(oa, fa, a, allr, ob, fb, b, allr, (tag, mode, F, H, t))
    assert a.device_error() == 0 and b.device_error() == 0
    tgs._release(a, b)


@pytest.mark.parametrize("tag", TAGS)
def test_primed_logits_within_the_oracle_bound(tag):
    """Default kernels, priming walk of the model's own time chunk choice: with H >= F the primed stream is a stream that
    received its clip from frame 0, so its logits hold to bound.model over that history."""
    a = tgs._model(tag)
    _, arch_fn = tgm.MODELS[tag]
    sd = tgm._oracle_state(a)
    arch = arch_fn(skeleton="kinetics" if bench.V == 18 else "ntu", classes=bench.CLASSES)
    xs = tgs._frames(N, 31)
    picks = tgs._picks()[:ORACLE_STREAMS]
    pk = torch.tensor(picks, device=DEV)
    ys = _history(picks, 32)
    F = a.delay + 5
    for t in range(F):
        a.forward_step(xs[t % 8])
    a.prime_streams(picks, torch.stack([ys[t % 8] for t in range(F)], dim=2))
    T = F + a.receptive_field + a.stride
    logits = []
    for t in range(F, T):
        out = a.forward_step(_feed(xs[t % 8], pk, ys, t))
        if out is not None:
            logits.append(out[pk].cpu())
    assert a.device_error() == 0
    tgs._release(a)
    got = torch.stack(logits, dim=2)
    with torch.no_grad():
        value, mag = bound.model(torch.stack([ys[t % 8].cpu() for t in range(T)], dim=2), sd, arch)
    n = got.shape[2]
    h = bound.headroom(got, value[:, :, -n:], len(arch.blocks) * mag[:, :, -n:])
    print(f"\n[prime] {tag}: {n} emissions after priming, logits max err/(10*EPS*mag) = {h:.3f}")
    assert h <= 1.0, (tag, h)


@pytest.mark.parametrize("tag", TAGS)
def test_refusals_leave_every_stream_alone(tag):
    a = tgs._model(tag)
    picks = tgs._picks()
    ys = _history(picks, 42)
    clip = torch.stack([ys[t % 8] for t in range(12)], dim=2)
    with pytest.raises(cs.CoskError):  # before the first step
        a.prime_streams(picks, clip)
    xs = tgs._frames(N, 41)
    F = 20
    for t in range(F):
        a.forward_step(xs[t % 8])
    before = _export_all(a)
    bad = [
        ([picks[0], picks[0]], clip[:2]),                     # repeat
        ([N], clip[:1]),                                      # out of range
        ([-1], clip[:1]),
        (picks, clip[:-1]),                                   # one clip row short
        (picks, clip[..., :-1]),                              # wrong V / S
        (picks, clip[:, :, 0]),                               # no time axis
        (picks, clip.cpu()),                                  # not on the device
    ]
    for idx, x in bad:
        with pytest.raises(cs.CoskError):
            a.prime_streams(idx, x)
        assert a.frame_count() == F
    assert torch.equal(_export_all(a), before)
    # a handle whose state no longer matches its weights is refused by the same entry check as a latched one
    e = a._engine
    idx = (ctypes.c_int64 * 1)(picks[0])
    w = torch.zeros(bench.CLASSES, dtype=torch.float32)
    assert e.lib.cosk_load_weights(e.h, b"fc.b", ctypes.c_void_p(w.data_ptr()), w.numel()) == 0
    assert e.lib.cosk_prime_streams(e.h, idx, 1, ctypes.c_void_p(clip.data_ptr()), 12, 1, None) == -3
    assert e.lib.cosk_frame_count(e.h) == F
    fresh = tgs._model(tag)
    fe = fresh._sync(torch.device(DEV))
    assert fe.lib.cosk_prime_streams(fe.h, idx, 1, ctypes.c_void_p(clip.data_ptr()), 12, 1, None) == -3
    tgs._release(a, fresh)


@pytest.mark.parametrize("tag", TAGS)
def test_launches_and_memory(tag, monkeypatch):
    """k = N and k = 1 at time chunk 16: the priming walk takes the launches forward_steps takes for the same frames, plus the
    gather and the scatter, and device memory returns to its level before the call.  With H >= receptive_field streams
    primed from the frames they already received come out bit-identical."""
    monkeypatch.setenv("COSK_FUSE_BLOCK", "0")
    a = tgs._model(tag, time_chunk=16)
    H = a.receptive_field + 3
    F = H + 7
    xs = tgs._frames(N, 51)
    for t in range(F - H):
        a.forward_step(xs[t % 8])
    clip = torch.stack([xs[t % 8] for t in range(F - H, F)], dim=2)
    n0 = a.launch_count()
    a.forward_steps(clip)
    steps_launches = a.launch_count() - n0
    assert a.frame_count() == F
    state = _export_all(a)
    a.prime_streams([N - 1], clip[N - 1:])  # loads the modules the call uses before memory is compared
    for idx in (list(range(N)), [N // 2]):
        sub = clip[idx]
        torch.cuda.synchronize()
        free0, _ = torch.cuda.mem_get_info()
        n0 = a.launch_count()
        a.prime_streams(idx, sub)
        assert a.launch_count() - n0 <= steps_launches + 2, (tag, len(idx), a.launch_count() - n0, steps_launches)
        assert torch.cuda.mem_get_info()[0] == free0, (tag, len(idx))
        assert torch.equal(_export_all(a), state), (tag, len(idx))
    n0 = a.launch_count()
    a.prime_streams([3], clip[:1, :, :0])  # H = 0: a reset, one launch
    assert a.launch_count() == n0 + 1
    tgs._release(a)


def test_multistream_members_stay_in_lock_step():
    tag = "cost_gcn"
    n = 64
    members = [tgs._model(tag, seed=s) for s in (0, 1)]
    solo = [tgs._twin(m, tag) for m in members]
    ens = cs.MultiStream(members)
    xs = [tgs._frames(n, 61 + i) for i in range(2)]
    F = 40
    for t in range(F):
        ens.forward_step([x[t % 8] for x in xs])
        for s, x in zip(solo, xs):
            s.forward_step(x[t % 8])
    picks = [5, 17]
    clips = [torch.stack([x[(t + 3) % 8][:2] for t in range(30)], dim=2) for x in xs]
    ens.prime_streams(picks, clips)
    for s, c in zip(solo, clips):
        s.prime_streams(picks, c)
    for m, s in zip(members, solo):
        assert m.frame_count() == s.frame_count() == F
        assert torch.equal(m.export_streams(list(range(n))).payload, s.export_streams(list(range(n))).payload)
    emitted = 0
    for t in range(F, members[0].delay + 2 * members[0].stride):
        out = ens.forward_step([x[t % 8] for x in xs])  # raises if the members fell out of lock step
        emitted += out is not None
    assert emitted > 0
    tgs._release(*members, *solo)
