"""Per-stream state without a GPU: the host-side schedule compatibility rule that import_streams applies, and MultiStream's
forwarding of the per-stream calls to its members."""
import ctypes

import numpy as np
import pytest

import continual_skeletons_b200 as cs
from continual_skeletons_b200 import lib as _lib

CONFIGS = {
    "cost_gcn": lambda: cs.CoStGcn({"dataset_name": "dummy_ntu"}),
    "cost_gcn_mod": lambda: cs.CoStGcnMod({"dataset_name": "dummy_ntu"}),
    "coa_gcn": lambda: cs.CoAGcn({"dataset_name": "ntu120", "forward_mode": "frame"}),
    "cos_tr": lambda: cs.CoSTr({"dataset_name": "dummy_kin"}),
}


@pytest.mark.parametrize("tag", list(CONFIGS))
def test_schedule_compatible_is_agreement_of_future_flags(tag):
    """For every pair of frame counts in [0, 2H): compatible iff the flags simulate_schedule gives from both agree over the
    next H frames, H = receptive field + stride (past the warm-up, and one more period of the strides)."""
    model = CONFIGS[tag]()
    lib = _lib.load_library()
    cfg = model._config()
    H = model.receptive_field + model.stride
    sched = np.array(model.simulate_schedule(3 * H), dtype=np.uint8)
    keys = {}
    window = np.array([keys.setdefault(sched[a: a + H].tobytes(), len(keys)) for a in range(2 * H)])
    want = window[:, None] == window[None, :]
    got = np.empty_like(want)
    fn = lib.cosk_schedule_compatible
    ref = ctypes.byref(cfg)
    for a in range(2 * H):
        for b in range(2 * H):
            got[a, b] = fn(ref, a, b) == 1
    assert np.array_equal(got, want), np.argwhere(got != want)[:8]
    # the rule in practice: equal, or both past the warm-up and congruent modulo the stride
    late = 2 * H - 1
    assert model.schedule_compatible(late, late - model.stride)
    assert model.schedule_compatible(10 ** 12, 10 ** 12 + 3 * model.stride)
    if model.stride > 1:
        assert not model.schedule_compatible(late, late - 1)
    assert not model.schedule_compatible(0, model.stride)


def test_schedule_compatible_rejects_bad_arguments():
    lib = _lib.load_library()
    cfg = CONFIGS["cost_gcn"]()._config()
    assert lib.cosk_schedule_compatible(ctypes.byref(cfg), -1, 0) == -1
    assert lib.cosk_schedule_compatible(None, 0, 0) == -1


class _Member:
    def __init__(self):
        self.calls = []
        self.receptive_field, self.stride, self.padding = 449, 4, 152

    def reset_streams(self, indices):
        self.calls.append(("reset_streams", list(indices)))

    def resize_streams(self, keep):
        self.calls.append(("resize_streams", list(keep)))


def test_multistream_forwards_per_stream_calls():
    members = [_Member(), _Member()]
    ens = cs.MultiStream(members)
    ens.reset_streams([3, 1])
    ens.resize_streams([0, -1, 2])
    for m in members:
        assert m.calls == [("reset_streams", [3, 1]), ("resize_streams", [0, -1, 2])]
