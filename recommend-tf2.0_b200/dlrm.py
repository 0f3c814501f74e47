"""DLRM with the reference's constructor (src/ctr/dlrm/model.py:16-40) on the B200 kernels.

The reference's `call` is broken (`self.dense_inputs`, `self.dnn_network` do not exist, :44,50)
and concatenates where the paper it cites interacts (:48).  `interaction='dot'` (default) is
the paper's pairwise dot through the fused gather+interaction kernel; `interaction='cat'`
reproduces line 48 literally.  Dense MLPs are framework GEMMs (fp32); embeddings, interaction,
their backward and the sparse optimizer are librtf_b200 kernels.
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch

from .embedding import EmbeddingTables, SparseOptimizer
from .interaction import dot_out_cols, embed_dot
from .core import DNN, Dense, DenseAdam, Layer, StepGraph, binary_crossentropy


class DLRM(Layer):
    def __init__(self, feature_columns, bot_dnn_hidden_units=(64, 32, 16),
                 top_dnn_hidden_units=(128, 64), activation="relu", dnn_dropout=0.0,
                 embed_reg=1e-4, interaction: str = "dot",
                 sparse_optimizer: Optional[SparseOptimizer] = None, pad_to: int = 1,
                 input_bn: bool = True, seed: Optional[int] = None):
        super().__init__()
        self.dense_feature_columns, self.sparse_feature_columns = feature_columns
        self.interaction, self.pad_to, self.embed_reg = interaction, pad_to, embed_reg
        rows = [f["feat_num"] for f in self.sparse_feature_columns]
        dims = [f["embed_dim"] for f in self.sparse_feature_columns]
        if interaction == "dot" and (len(set(dims)) != 1 or bot_dnn_hidden_units[-1] != dims[0]):
            raise ValueError("dot interaction needs equal embed_dim == bot_dnn_hidden_units[-1]")
        # 'random_uniform' + l2(embed_reg) as at model.py:31-35
        self.embed_layers = EmbeddingTables(rows, dims, "random_uniform",
                                            optimizer=sparse_optimizer, seed=seed)
        self.bot_dnn = DNN(bot_dnn_hidden_units, activation, dnn_dropout, input_bn=input_bn)
        self.top_dnn = DNN(top_dnn_hidden_units, activation, dnn_dropout, input_bn=input_bn)
        self.final_dense = Dense(1, activation=None)

    def call(self, inputs, **kwargs):
        dense_inputs, sparse_inputs = inputs
        dense_fea = self.bot_dnn(dense_inputs)
        if self.interaction == "cat":
            sparse_embed = self.embed_layers.lookup(sparse_inputs)
            x = torch.cat([sparse_embed, dense_fea], dim=-1)
        else:
            x = embed_dot(self.embed_layers, sparse_inputs, dense_fea, pad_to=self.pad_to)
        top = self.final_dense(self.top_dnn(x))
        return torch.sigmoid(top)

    def dense_parameters(self):
        emb = {id(p) for p in self.embed_layers.parameters()}
        return [p for p in self.parameters() if id(p) not in emb]


def build_dense_layers(model, n_dense: int, device, n_tables: Optional[int] = None) -> None:
    """Create the lazily built MLP weights (Keras layers build on first call) WITHOUT running the
    model: a 4-row zero batch through the bottom / top stacks in eval mode (BatchNorm's moving
    statistics do not move); none of the embedding-path kernels run."""
    was_training = model.training
    model.eval()
    with torch.no_grad():
        d = model.bot_dnn(torch.zeros(4, n_dense, device=device))
        if getattr(model, "interaction", "dot") == "cat":
            cols = sum(int(w.shape[1]) for w in model.embed_layers.weights) + d.shape[1]
        else:
            if n_tables is None:
                n_tables = len(model.embed_layers.weights)
            cols = dot_out_cols(n_tables + 1, d.shape[1], model.pad_to)
        model.final_dense(model.top_dnn(torch.zeros(4, cols, device=device)))
    model.train(was_training)


class DLRMTrainer:
    """One training step = forward, Keras BCE, backward (K4 bwd -> K2 with the fused sparse
    optimizer on the tables), dense Adam on the MLPs (Keras form, core.DenseAdam: one
    rtf_dense_adam launch over the flat parameter buffer)."""

    def __init__(self, model: DLRM, lr: float = 1e-3, cuda_graph: bool = False, metrics=None):
        self.model = model
        self.metrics = list(metrics or [])      # updated by every step (metrics.AUC)
        self.cuda_graph = cuda_graph
        self._evaluator = None
        if model.embed_layers.optimizer is None:
            model.embed_layers.set_optimizer(SparseOptimizer("adam", lr=lr, l2=model.embed_reg))
        self.dense_opt = None
        self.lr = lr
        model.embed_layers.async_update = True     # the step ends with wait_pending()
        # cuda_graph: replay the step from a CUDA graph (core.StepGraph); pays off when the step is
        # launch-bound (small batches) — at batch 65536 the GPU is the bound and it changes nothing
        self.graph = StepGraph(self._body, self._advance) if cuda_graph else None

    def _advance(self):
        self.model.embed_layers.begin_step()
        self.dense_opt.advance()

    def _body(self, inputs, labels):
        m = self.model
        pred = m(inputs)
        loss = binary_crossentropy(labels, pred)
        for mt in self.metrics:
            mt.update_state(labels, pred.detach())
        self.dense_opt.zero_grad()
        loss.backward()
        self.dense_opt.apply()
        m.embed_layers.wait_pending()   # K2's row update ran on the side stream behind the MLP backward
        return loss.detach()

    def _setup(self, dense):
        m = self.model
        if self.dense_opt is None:      # layers build on first call: build them, then flatten
            build_dense_layers(m, dense.shape[1], dense.device)
            self.dense_opt = DenseAdam(m.dense_parameters(), lr=self.lr)
            if self.graph is not None:
                self.dense_opt.enable_device_lr()
                m.embed_layers.optimizer.enable_device_lr(dense.device)

    def step(self, dense, sparse, labels) -> torch.Tensor:
        self._setup(dense)
        if self.graph is not None:
            return self.graph([dense, sparse], labels)
        self._advance()
        return self._body([dense, sparse], labels)

    def _eval_forward(self, inputs, labels):
        pred = self.model(inputs)
        return pred, binary_crossentropy(labels, pred)

    def evaluate(self, batches) -> dict:
        """Keras `model.evaluate` over `(dense, sparse, labels)` batches (as DeviceFeeder yields
        them): {"loss": batch-size-weighted mean BCE, <metric name>: value, ...}, computed by
        fresh copies of the trainer's metrics.  Changes no parameter, buffer, table, optimizer
        state or step counter (metrics.Evaluator)."""
        if self._evaluator is None:
            from .metrics import Evaluator
            self._evaluator = Evaluator(self._eval_forward, self.metrics, self.cuda_graph)
        pairs = (([dense, sparse], labels) for dense, sparse, labels in batches)
        return self._evaluator.run(self.model, pairs, lambda inputs: self._setup(inputs[0]))
