"""f4: weights round-trip under the Keras variable names of the reference's models (CPU)."""
import os

import numpy as np
import pytest
import torch

import recommend_tf2_b200 as pkg
from recommend_tf2_b200 import checkpoint as ck
from recommend_tf2_b200 import core
from recommend_tf2_b200.core import DNN, Dense, Layer
from recommend_tf2_b200.embedding import EmbeddingTables


@pytest.fixture(autouse=True)
def _layers_on_cpu(monkeypatch):
    """Layers create their weights on CUDA when a device is present; the model here runs on CPU
    tensors, so it is built on the CPU on every machine."""
    monkeypatch.setattr(core, "_default_device", lambda: torch.device("cpu"))


class TinyDLRM(Layer):
    """The reference DLRM's variable structure (src/ctr/dlrm/model.py:30-40): per-field
    Embedding layers, bottom DNN, top DNN, final Dense — on CPU tensors (no kernel runs)."""

    def __init__(self):
        super().__init__()
        self.embed_layers = EmbeddingTables([7, 5, 3], [4, 4, 4], device="cpu", seed=None)
        self.bot_dnn = DNN((8, 4))
        self.top_dnn = DNN((6,))
        self.final_dense = Dense(1)

    def call(self, x, **kwargs):
        return self.final_dense(self.top_dnn(self.bot_dnn(x)[:, :4].repeat(1, 3)[:, :10]))


def _build():
    torch.manual_seed(0)
    m = TinyDLRM()
    m.eval()
    with torch.no_grad():
        m(torch.rand(5, 13))
    return m


def test_names_follow_keras_auto_naming():
    names = list(ck.weights_dict(_build()).keys())
    assert names[:3] == ["embedding/embeddings:0", "embedding_1/embeddings:0", "embedding_2/embeddings:0"]
    # DNN = BatchNormalization created in call + Dense stack (src/ctr/layers/modules.py:129-135)
    assert "dense/kernel:0" in names and "dense/bias:0" in names and "dense_1/kernel:0" in names
    assert "batch_normalization/moving_variance:0" in names and "batch_normalization_1/gamma:0" in names
    assert names[-2:] == ["dense_3/kernel:0", "dense_3/bias:0"]
    assert len(names) == len(set(names)) == 3 + 2 * 4 + 4 * 2


def test_save_load_round_trip(tmp_path):
    a, b = _build(), _build()
    with torch.no_grad():
        for p in a.parameters():
            p.add_(torch.randn_like(p))
        a.bot_dnn.bn.moving_mean.add_(1.5)
    path = os.path.join(tmp_path, "dlrm_weights.epoch_0005")
    ck.save_weights(a, path)
    ck.load_weights(b, path)
    wa, wb = ck.weights_dict(a), ck.weights_dict(b)
    assert list(wa) == list(wb)
    for k in wa:
        assert np.array_equal(wa[k], wb[k]), k
    x = torch.rand(6, 13)
    with torch.no_grad():
        assert torch.equal(a(x), b(x))


def test_strict_name_check_and_prefix():
    m = _build()
    d = ck.weights_dict(m, prefix="dlrm/")
    assert all(k.startswith("dlrm/") for k in d)
    ck.set_weights_dict(m, d, prefix="dlrm/")
    bad = dict(d)
    bad.pop("dlrm/dense/bias:0")
    try:
        ck.set_weights_dict(m, bad, prefix="dlrm/")
        raise AssertionError("a missing variable must be reported")
    except KeyError:
        pass
    assert hasattr(pkg, "checkpoint") or True
