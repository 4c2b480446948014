"""On-device fusion of the per-modality models' logits ("multi-stream" evaluation).

The reference fuses the joint / bone / motion models offline: every model writes its logits to a ``.npy``
file and ``scripts/multi_stream_eval.py:33-42`` (``aggregate_preds``) reduces the files with ``np.add`` (or
``np.maximum``).  Online, the same reduction is applied to the logits of continual models that advance in lock
step on the same frames, without leaving the device.  All members must share the step schedule (same
architecture family), so they emit on the same frames.
"""
import torch

_METHODS = {"add": torch.add, "max": torch.maximum}


def aggregate_preds(preds, method="add"):
    """``aggregate_preds`` of scripts/multi_stream_eval.py:33-42 on device tensors (same shape check)."""
    if method not in _METHODS:
        raise ValueError(f"method must be one of {sorted(_METHODS)}")
    preds = list(preds)
    shapes = {tuple(p.shape) for p in preds}
    if len(shapes) != 1:
        raise ValueError(f"All preds should have the same shape but got {[tuple(p.shape) for p in preds]}")
    out = preds[0]
    for p in preds[1:]:
        out = _METHODS[method](out, p)
    return out


class MultiStream:
    """Lock-step ensemble of continual models, one per input modality (joint, bone, ...)."""

    def __init__(self, models, method="add"):
        self.models = list(models)
        if not self.models:
            raise ValueError("MultiStream needs at least one model")
        if method not in _METHODS:
            raise ValueError(f"method must be one of {sorted(_METHODS)}")
        sched = {(m.receptive_field, m.stride, m.padding) for m in self.models}
        if len(sched) != 1:
            raise ValueError("all member models must share receptive field, stride and padding")
        self.method = method

    def clean_state(self):
        for m in self.models:
            m.clean_state()

    def reset_streams(self, indices):
        """``reset_streams`` on every member: the listed streams start over in all modalities."""
        for m in self.models:
            m.reset_streams(indices)

    def resize_streams(self, keep):
        """``resize_streams`` on every member, so the members stay in lock step on the same streams."""
        for m in self.models:
            m.resize_streams(keep)

    def prime_streams(self, indices, clips):
        """``prime_streams`` on every member, member i from ``clips[i]`` (its modality of the same frames), so the members
        stay in lock step."""
        clips = list(clips)
        if len(clips) != len(self.models):
            raise ValueError(f"expected {len(self.models)} clips, got {len(clips)}")
        for m, clip in zip(self.models, clips):
            m.prime_streams(indices, clip)

    def forward_step(self, inputs):
        """inputs: one (N, C, V, S) CUDA tensor per member model.  Fused logits, or None when no prediction is due."""
        inputs = list(inputs)
        if len(inputs) != len(self.models):
            raise ValueError(f"expected {len(self.models)} inputs, got {len(inputs)}")
        outs = [m.forward_step(x) for m, x in zip(self.models, inputs)]
        if all(o is None for o in outs):
            return None
        if any(o is None for o in outs):
            raise RuntimeError("member models fell out of lock step (were some of them stepped separately?)")
        return aggregate_preds(outs, self.method)

    def forward_steps(self, inputs):
        """inputs: one (N, C, T, V, S) tensor per member; (N, classes, n_out) fused logits or None."""
        inputs = list(inputs)
        if len(inputs) != len(self.models):
            raise ValueError(f"expected {len(self.models)} inputs, got {len(inputs)}")
        outs = [m.forward_steps(x) for m, x in zip(self.models, inputs)]
        if all(o is None for o in outs):
            return None
        if any(o is None for o in outs):
            raise RuntimeError("member models fell out of lock step (were some of them stepped separately?)")
        return aggregate_preds(outs, self.method)
