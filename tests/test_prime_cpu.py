"""prime_streams without a GPU: MultiStream hands each member its own clip, and a model without stream state refuses."""
import pytest

import continual_skeletons_b200 as cs


class _Member:
    def __init__(self):
        self.calls = []
        self.receptive_field, self.stride, self.padding = 449, 4, 152

    def prime_streams(self, indices, clip):
        self.calls.append((list(indices), clip))


def test_multistream_primes_each_member_from_its_clip():
    members = [_Member(), _Member()]
    ens = cs.MultiStream(members)
    ens.prime_streams([3, 1], ["joint", "bone"])
    assert members[0].calls == [([3, 1], "joint")]
    assert members[1].calls == [([3, 1], "bone")]
    with pytest.raises(ValueError):
        ens.prime_streams([0], ["joint"])
    assert len(members[0].calls) == 1


@pytest.mark.parametrize("cls", [cs.CoStGcn, cs.CoStack])
def test_prime_before_any_step_is_refused(cls):
    model = cls({"dataset_name": "dummy_ntu"}) if cls is cs.CoStGcn else cls([(3, 64, 1, False)])
    with pytest.raises(cs.CoskError):
        model.prime_streams([0], None)
