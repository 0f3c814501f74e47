"""Keras-compatible metrics on the GPU: `AUC`, the metric every CTR script of the reference
compiles its model with (`model.compile(..., metrics=[AUC()])`, src/ctr/fm/train.py:50) and the
number it prints after `model.evaluate` (:58,67).

State lives in device memory and is updated by librtf_b200 kernels (csrc/metrics.cu): an update
is one launch and never synchronises, so it can run inside a training step, including one
replayed from a CUDA graph.  Semantics: SURVEY.md App. A19; divergences from Keras: DESIGN.md §3."""
from __future__ import annotations

import torch

from . import _lib as L

MAX_THRESHOLDS = 4096


class AUC:
    """tf.keras.metrics.AUC with its defaults: ROC curve, trapezoid ('interpolation') summation,
    `num_thresholds` evenly spaced thresholds.  Counts are exact int64 per threshold bucket.

        auc = AUC()
        auc.update_state(y_true, y_pred)     # (B, 1) or (B,) CUDA tensors, y_pred fp32 in [0, 1]
        auc.result()                         # 0-d fp32 device tensor
        auc.check()                          # raises ValueError if an update saw invalid input
    """

    def __init__(self, num_thresholds: int = 200, curve: str = "ROC",
                 summation_method: str = "interpolation", name: str = "auc"):
        if curve != "ROC":
            raise ValueError(f"AUC: curve={curve!r} is not supported (only 'ROC')")
        if summation_method != "interpolation":
            raise ValueError(f"AUC: summation_method={summation_method!r} is not supported "
                             "(only 'interpolation')")
        if not 2 <= int(num_thresholds) <= MAX_THRESHOLDS:
            raise ValueError(f"AUC: num_thresholds must be in [2, {MAX_THRESHOLDS}], "
                             f"got {num_thresholds}")
        self.num_thresholds, self.curve = int(num_thresholds), curve
        self.summation_method, self.name = summation_method, name
        self.counts = None      # (2, T) int64: per-bucket positives, negatives
        self.err = None         # (1,) int32: bit 0 = an update saw invalid input

    def get_config(self) -> dict:
        return {"num_thresholds": self.num_thresholds, "curve": self.curve,
                "summation_method": self.summation_method, "name": self.name}

    def build(self, device) -> None:
        """Allocate the state on `device` (done by the first update).  A CUDA graph that updates
        the metric holds these addresses: they never change afterwards."""
        if self.counts is None:
            self.counts = torch.zeros((2, self.num_thresholds), dtype=torch.int64, device=device)
            self.err = torch.zeros(1, dtype=torch.int32, device=device)

    def update_state(self, y_true: torch.Tensor, y_pred: torch.Tensor) -> None:
        L.require_cuda(y_pred, "AUC.update_state(y_pred)")
        L.require_cuda(y_true, "AUC.update_state(y_true)")
        if y_pred.dtype != torch.float32:
            raise TypeError("AUC.update_state: y_pred must be fp32")
        p = y_pred.reshape(-1).contiguous()
        y = y_true.to(torch.float32).reshape(-1).contiguous()
        if p.numel() != y.numel():
            raise ValueError(f"AUC.update_state: {y.numel()} labels for {p.numel()} predictions")
        self.build(p.device)
        if p.numel() == 0:      # an empty tensor has no storage pointer; nothing to count
            return
        L.check(L.lib().rtf_auc_update(p.data_ptr(), y.data_ptr(), p.numel(), self.num_thresholds,
                                       self.counts.data_ptr(), self.err.data_ptr(),
                                       L.current_stream_ptr()), "rtf_auc_update")

    def result(self) -> torch.Tensor:
        if self.counts is None:
            raise L.RtfError("AUC.result: no state yet (update_state first); the metric lives "
                             "on a CUDA device")
        out = torch.empty((), dtype=torch.float32, device=self.counts.device)
        L.check(L.lib().rtf_auc_result(self.counts.data_ptr(), self.num_thresholds, out.data_ptr(),
                                       L.current_stream_ptr()), "rtf_auc_result")
        return out

    def reset_state(self) -> None:
        """Zero the counts and the error flag IN PLACE (a captured graph holds their addresses)."""
        if self.counts is not None:
            self.counts.zero_()
            self.err.zero_()

    def check(self) -> None:
        """Raise ValueError if any update since the last reset saw a prediction outside [0, 1]
        (or NaN) or a label other than 0 / 1 — Keras raises on such input.  Synchronises."""
        if self.err is not None and int(self.err.item()) != 0:
            raise ValueError(f"{self.name}: predictions must be in [0, 1] and labels 0 or 1; "
                             "invalid elements were not counted")


class Evaluator:
    """The evaluation loop of `Trainer.evaluate` / `DLRMTrainer.evaluate` (Keras `model.evaluate`):
    for each batch the model runs in eval() mode under no_grad (BatchNorm uses its moving
    statistics), loss * B is added to an fp64 device accumulator (Keras' batch-size-weighted
    mean) and the metrics are updated.  One host synchronisation at the end.

    The metrics are copies of the trainer's (same configuration, own state, reset at every run),
    so training-time state is untouched.  With cuda_graph=True the batches are replayed from a
    CUDA graph (core.StepGraph with nothing to advance); a batch of another shape runs eagerly."""

    def __init__(self, forward, metrics, cuda_graph: bool = False):
        from .core import StepGraph
        self.forward = forward      # (inputs, labels) -> (predictions, scalar loss)
        self.metrics = [type(m)(**m.get_config()) for m in metrics]
        self.acc = None
        self.graph = StepGraph(self._body, lambda: None) if cuda_graph else None

    def _body(self, inputs, labels):
        pred, loss = self.forward(inputs, labels)
        B = _first_leaf(inputs).shape[0]
        self.acc.add_(loss.to(torch.float64), alpha=B)
        for m in self.metrics:
            m.update_state(labels, pred)
        return loss

    def run(self, model, batches, prepare) -> dict:
        """batches: iterable of (inputs, labels); prepare(inputs) runs before the first batch."""
        was = model.training
        n, first = 0, True
        try:
            for inputs, labels in batches:
                if first:
                    first = False
                    prepare(inputs)
                    dev = _first_leaf(inputs).device
                    if self.acc is None:
                        self.acc = torch.zeros((), dtype=torch.float64, device=dev)
                    self.acc.zero_()
                    for m in self.metrics:
                        m.build(dev)
                        m.reset_state()
                    model.eval()
                with torch.no_grad():
                    if self.graph is not None:
                        self.graph(inputs, labels)
                    else:
                        self._body(inputs, labels)
                n += _first_leaf(inputs).shape[0]
        finally:
            model.train(was)
        if first:
            raise ValueError("evaluate: no batches")
        vals = torch.stack([self.acc / n] + [m.result().to(torch.float64)
                                             for m in self.metrics]).tolist()
        for m in self.metrics:
            m.check()
        out = {"loss": vals[0]}
        out.update((m.name, v) for m, v in zip(self.metrics, vals[1:]))
        return out


def _first_leaf(x):
    while isinstance(x, (list, tuple)):
        x = x[0]
    return x
