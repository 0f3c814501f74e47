"""The callers either side of the hot path: the reference's model classes (L3) rebuilt on the
drop-in layers, with the reference's constructor signatures.  Where the reference's `call` is
broken (SURVEY.md §0) the layer code is followed and the glue is defined here; every such
place is marked.  Dense MLP pieces are framework GEMMs (core.py)."""
from __future__ import annotations

from typing import Optional

import torch

from .embedding import EmbeddingTables, SparseOptimizer
from .layers.core import DNN, BatchNormalization, Dense, Dropout, Layer
from .layers.ctr import FM, AttentionLayer
from .layers.ctr import MultiHeadAttention as CtrMultiHeadAttention
from .layers.embedding import _as_int_ids
from .layers.match import DNN as MatchDNN
from .layers.match import SampledSoftmaxLayer, TransformerEncoder


class DeepFM(Layer):
    """src/ctr/deep_fm/model.py:17-65.  Embeddings use 'random_normal' (:35); the FM layer gets
    first_inputs = concat(dense, sparse_embed) and the 2-D sparse_embed as second_inputs
    (:56-59), exactly as the source does."""

    def __init__(self, feature_columns, hidden_units=(128, 64, 32), dnn_dropout=0.0,
                 activation="relu", fm_w_reg=1e-6, embed_reg=1e-6,
                 sparse_optimizer: Optional[SparseOptimizer] = None, seed=None):
        super().__init__()
        self.dense_feature_columns, self.sparse_feature_columns = feature_columns
        rows = [f["feat_num"] for f in self.sparse_feature_columns]
        dims = [f["embed_dim"] for f in self.sparse_feature_columns]
        self.embed_layers = EmbeddingTables(rows, dims, "random_normal", optimizer=sparse_optimizer,
                                            seed=seed)
        self.feature_length = len(self.dense_feature_columns) + sum(dims)
        self.fm = FM(self.feature_length, fm_w_reg)
        self.dnn = DNN(hidden_units, activation, dnn_dropout)
        self.dense = Dense(1, activation=None)

    def call(self, inputs, **kwargs):
        dense_inputs, sparse_inputs = inputs
        sparse_embed = self.embed_layers.lookup(_as_int_ids(sparse_inputs))      # (B, F*D)
        embeds = torch.cat([dense_inputs, sparse_embed], dim=-1)
        fm_outputs = self.fm([embeds, sparse_embed])                              # (B, 1)
        deep_outputs = self.dense(self.dnn(embeds))                               # (B, 1)
        return torch.sigmoid(fm_outputs + deep_outputs)


class AutoInt(Layer):
    """AutoInt on (B, F, d) field embeddings: `n_layers` stacked interacting layers
    (ctr MultiHeadAttention, use_res=True), flatten, Dense(1), sigmoid.

    The reference's AutoInt (src/ctr/autoint/model.py:44-55) feeds a 2-D (B, 26*D+13) tensor
    into the attention layer (batch-folding bug) with one layer / one head; BASELINE's config
    (3 layers, 2 heads, 39 fields, d=16) needs the paper's dense-field embedding x_j * v_j, which
    is defined here (SURVEY §0): `dense_embed` holds one d-vector per dense feature."""

    def __init__(self, feature_columns, head_size=16, head_num=2, n_layers=3, use_res=True,
                 activation="relu", embed_reg=1e-4, scale="reference",
                 sparse_optimizer: Optional[SparseOptimizer] = None, seed=None):
        super().__init__()
        self.dense_feature_columns, self.sparse_feature_columns = feature_columns
        rows = [f["feat_num"] for f in self.sparse_feature_columns]
        dims = [f["embed_dim"] for f in self.sparse_feature_columns]
        assert len(set(dims)) == 1
        self.d = dims[0]
        self.embed_layers = EmbeddingTables(rows, dims, "random_uniform", optimizer=sparse_optimizer,
                                            seed=seed)
        nd = len(self.dense_feature_columns)
        self.dense_embed = torch.nn.Parameter(
            torch.empty(nd, self.d, device=self.embed_layers.weights[0].device).uniform_(-0.05, 0.05))
        self.att_layers = torch.nn.ModuleList(
            [CtrMultiHeadAttention(head_size, head_num, activation=activation, use_res=use_res,
                                   scale=scale) for _ in range(n_layers)])
        self.out_dense = Dense(1, activation=None)

    def call(self, inputs, **kwargs):
        dense_inputs, sparse_inputs = inputs
        B, F = sparse_inputs.shape
        sparse_embed = self.embed_layers.lookup(_as_int_ids(sparse_inputs)).reshape(B, F, self.d)
        dense_embed = dense_inputs.unsqueeze(-1) * self.dense_embed.unsqueeze(0)   # x_j * v_j
        x = torch.cat([dense_embed, sparse_embed], dim=1)                          # (B, 39, d)
        for layer in self.att_layers:
            x = layer(x)
        return torch.sigmoid(self.out_dense(x.reshape(B, -1)))


class DIN(Layer):
    """DIN with the local activation unit on the classic input the reference's loader produces
    (src/ctr/utils/data_process.py:176,215-216): hist (B, maxlen, n_behavior) ids, target item
    (B, n_behavior) ids sharing the item tables (src/ctr/din/model.py:71-72), a (B, maxlen) mask
    = (hist[..., 0] != 0).  The reference's DIN.call never reaches a loss (reshape bug :79-81)
    and uses self-attention instead of AttentionLayer; this follows the layer + the paper."""

    def __init__(self, behavior_feature_nums, embed_dim=8, att_activation="sigmoid",
                 ffn_hidden_units=(80, 40), maxlen=100, dnn_dropout=0.0, embed_reg=1e-4,
                 sparse_optimizer: Optional[SparseOptimizer] = None, seed=None):
        super().__init__()
        nb = len(behavior_feature_nums)
        self.nb, self.embed_dim, self.maxlen = nb, embed_dim, maxlen
        self.embed_layers = EmbeddingTables(list(behavior_feature_nums), [embed_dim] * nb,
                                            "random_uniform", optimizer=sparse_optimizer, seed=seed)
        self.attention_layer = AttentionLayer(1, activation=att_activation)
        self.bn = BatchNormalization()
        self.ffn = torch.nn.ModuleList([Dense(u, activation="relu") for u in ffn_hidden_units])
        self.dropout = Dropout(dnn_dropout)
        self.final_output = Dense(1)

    def call(self, inputs, **kwargs):
        hist, target = inputs                       # (B, L, nb) ids, (B, nb) ids
        hist, target = _as_int_ids(hist), _as_int_ids(target)
        tabs = tuple(range(self.nb))
        k = self.embed_layers.lookup(hist, tabs, "BLF")            # (B, L, nb*D) — shared tables
        q = self.embed_layers.lookup(target, tabs, "BF")           # (B, nb*D)
        mask = (hist[..., 0] != 0).to(torch.float32)
        user_info = self.attention_layer([q, k, k, mask])
        x = self.bn(torch.cat([user_info, q], dim=-1))
        for dense in self.ffn:
            x = dense(x)
        return torch.sigmoid(self.final_output(self.dropout(x)))


class _SasrecScoreFn(torch.autograd.Function):
    """a10 epilogue (csrc/sasrec_score.cu): pos / neg gathers + dot scores + the log loss in one
    launch; backward re-gathers, returns d seq_info and hands the row gradients to K2."""

    @staticmethod
    def forward(ctx, tset: EmbeddingTables, info, pos, neg, pos_t, neg_t, *weights):
        import ctypes as C
        from . import _lib as L
        from .fm import colsum
        L.require_cuda(info, "SASRec scores(seq_info)")
        info = info.contiguous()
        pos, neg = pos.reshape(-1).contiguous(), neg.contiguous()
        if pos.dtype != neg.dtype:
            neg = neg.to(pos.dtype)
        B, D = info.shape
        NEG = neg.shape[1]
        Wp, Wn = weights[pos_t], weights[neg_t]
        logits = torch.empty((B, 1 + NEG), dtype=torch.float32, device=info.device)
        rows = torch.empty((B, 1), dtype=torch.float32, device=info.device)
        rc = L.lib().rtf_sasrec_score_fwd(info.data_ptr(), info.stride(0), Wp.data_ptr(), Wp.shape[0],
                                          Wn.data_ptr(), Wn.shape[0], pos.data_ptr(), neg.data_ptr(),
                                          int(pos.dtype == torch.int64), neg.stride(0), B, NEG, D,
                                          logits.data_ptr(), rows.data_ptr(), tset.err.data_ptr(),
                                          L.current_stream_ptr())
        L.check(rc, "rtf_sasrec_score_fwd")
        loss = colsum(rows).reshape(()) / (2.0 * B * NEG)
        ctx.tset, ctx.tabs = tset, (pos_t, neg_t)
        ctx.save_for_backward(info, pos, neg, logits)
        return logits, loss

    @staticmethod
    def backward(ctx, glogits, gloss):
        from . import _lib as L
        info, pos, neg, logits = ctx.saved_tensors
        tset, (pos_t, neg_t) = ctx.tset, ctx.tabs
        Wp, Wn = tset.weights[pos_t], tset.weights[neg_t]
        B, D = info.shape
        NEG = neg.shape[1]
        ginfo = torch.empty_like(info)
        gemb = torch.empty((B, 1 + NEG, D), dtype=torch.float32, device=info.device)
        gl = None if gloss is None else gloss.reshape(1).to(torch.float32).contiguous()
        gg = None if glogits is None else glogits.contiguous()
        rc = L.lib().rtf_sasrec_score_bwd(info.data_ptr(), info.stride(0), Wp.data_ptr(), Wp.shape[0],
                                          Wn.data_ptr(), Wn.shape[0], pos.data_ptr(), neg.data_ptr(),
                                          int(pos.dtype == torch.int64), neg.stride(0), B, NEG, D,
                                          logits.data_ptr(), None if gl is None else gl.data_ptr(),
                                          None if gg is None else gg.data_ptr(), ginfo.data_ptr(),
                                          gemb.data_ptr(), L.current_stream_ptr())
        L.check(rc, "rtf_sasrec_score_bwd")
        # row gradients -> K2 (fused sparse optimizer, or sparse COO gradients per table)
        nw = len(tset.weights)
        g_pos = tset.grads_from_lookup_grad(pos.reshape(B, 1), (pos_t,), gemb[:, 0, :], "BL", None)
        g_neg = tset.grads_from_lookup_grad(neg, (neg_t,), gemb[:, 1:, :], "BL", None)
        wg = [None] * nw
        for g, t in ((g_pos, pos_t), (g_neg, neg_t)):      # only the tables that were looked up
            if g[t] is not None:
                wg[t] = g[t] if wg[t] is None else wg[t] + g[t]
        return (None, ginfo, None, None, None, None) + tuple(wg)


class SASRec(Layer):
    """src/match/sasrec/model.py:19-97: three separate tables (seq/pos/neg item, :75-79), no
    positional embedding (:74), x *= mask before and after every block (:82,86), last position,
    dot scores and the log loss (:88-95).  Returns (logits (B, 1+neg_len), loss)."""

    def __init__(self, item_num, embed_dim=64, blocks=2, num_heads=1, ffn_hidden_unit=128,
                 dropout=0.0, seq_len=10, neg_len=100, layer_norm_eps=1e-6,
                 sparse_optimizer: Optional[SparseOptimizer] = None, seed=None):
        super().__init__()
        self.seq_len, self.neg_len, self.embed_dim = seq_len, neg_len, embed_dim
        self.fused_scores = True    # False: separate lookups + framework elementwise tail
        self.tables = EmbeddingTables([item_num] * 3, [embed_dim] * 3, "random_uniform",
                                      optimizer=sparse_optimizer, seed=seed)
        self.encoder_layer = torch.nn.ModuleList(
            [TransformerEncoder(embed_dim, num_heads, ffn_hidden_unit, dropout, layer_norm_eps)
             for _ in range(blocks)])

    def call(self, inputs, **kwargs):
        seq, pos, neg = (_as_int_ids(t) for t in inputs)     # (B,L), (B,1), (B,neg_len)
        mask = (seq != 0).to(torch.float32).unsqueeze(-1)                       # :72
        seq_embed = self.tables.lookup(seq, (0,), "BL")                         # (B,L,D)
        att_outputs = seq_embed * mask                                          # :81-82
        for block in self.encoder_layer:
            att_outputs = block([att_outputs, mask])
            att_outputs = att_outputs * mask                                    # :86
        if self.fused_scores:
            # :77-79 + :88-96 in one launch (the pos / neg rows never round-trip HBM)
            return _SasrecScoreFn.apply(self.tables, att_outputs[:, -1, :], pos, neg, 1, 2,
                                        *self.tables.weights)
        pos_embed = self.tables.lookup(pos, (1,), "BL")
        neg_embed = self.tables.lookup(neg, (2,), "BL")
        seq_info = att_outputs[:, -1:, :]                                       # :88
        pos_scores = (seq_info * pos_embed).sum(-1)
        neg_scores = (seq_info * neg_embed).sum(-1)
        loss = (-torch.log(torch.sigmoid(pos_scores)) -
                torch.log(1 - torch.sigmoid(neg_scores))).mean() / 2           # :93-95
        return torch.cat([pos_scores, neg_scores], dim=-1), loss


class YoutubeDNN(Layer):
    """Two towers + sampled softmax.  conventional=True (BASELINE config): the class weights are
    an item table (item_num, D) and num_classes = item_num.  conventional=False reproduces
    src/match/youtube_dnn/model.py:43-61 literally (weights = in-batch item tower output,
    num_classes = tower width)."""

    def __init__(self, user_feature_nums, item_num, embed_dim=64, user_dnn_hidden_units=(64, 32),
                 num_sampled=5, conventional=True, sparse_optimizer: Optional[SparseOptimizer] = None,
                 seed=None):
        super().__init__()
        self.conventional, self.num_sampled, self.item_num = conventional, num_sampled, item_num
        nu = len(user_feature_nums)
        self.user_tables = EmbeddingTables(list(user_feature_nums), [embed_dim] * nu,
                                           optimizer=sparse_optimizer, seed=seed)
        width = user_dnn_hidden_units[-1]
        self.item_table = EmbeddingTables([item_num], [width if conventional else embed_dim],
                                          optimizer=sparse_optimizer if conventional else None,
                                          seed=seed)
        self.user_dnn = MatchDNN(user_dnn_hidden_units)
        self.item_dnn = None if conventional else MatchDNN(user_dnn_hidden_units)
        self.sampler_layer = SampledSoftmaxLayer(num_sampled)
        self._step = 0
        self.seed_dev = None

    def enable_device_seed(self, device):
        """The sampler's per-step seed (the step counter) in device memory, bumped by advance():
        the candidate draw then changes on every replay of a captured step (core.StepGraph).
        Same seeds, hence the same candidates, as the host-seeded path."""
        if self.seed_dev is None:
            self.seed_dev = torch.full((1,), self._step, dtype=torch.int64, device=device)

    def advance(self):
        self._step += 1
        self.seed_dev.fill_(self._step)

    def call(self, inputs, sampled_values=None, **kwargs):
        from .layers.match import sampled_softmax_loss
        user_ids, item_ids = (_as_int_ids(t) for t in inputs[:2])
        user_out = self.user_dnn(self.user_tables.lookup(user_ids))             # (B, width)
        if self.seed_dev is None:
            self._step += 1
        if self.conventional:
            loss = sampled_softmax_loss(self.item_table.weights[0], None, item_ids, user_out,
                                        self.num_sampled, self.item_num,
                                        sampled_values=sampled_values,
                                        seed=self._step if self.seed_dev is None else self.seed_dev,
                                        err=self.item_table.err, table=(self.item_table, 0))
            return loss.unsqueeze(1)
        item_out = self.item_dnn(self.item_table.lookup(item_ids.reshape(-1, 1)))
        labels = inputs[2]
        return self.sampler_layer([item_out.unsqueeze(1), user_out.unsqueeze(1), labels],
                                  sampled_values=sampled_values)


class Trainer:
    """model.compile(loss, optimizer=Adam(lr)) + one fit step (src/ctr/fm/train.py:49-50,57-64)
    for any model of this module: embedding tables are updated in place by K2's fused sparse
    Adam during the backward, every other parameter by one rtf_dense_adam launch (Keras form).

        tr = Trainer(model, loss_fn, metrics=[AUC()])   # loss_fn(outputs, labels) -> scalar
        loss = tr.step(inputs, labels)        # also updates tr.metrics (inside the graph too)
        tr.evaluate([(inputs, labels), ...])  # {"loss": ..., "auc": ...}, Keras model.evaluate

    The lazily built layers are created by a no-grad eval forward on the first batch (BatchNorm
    moving statistics and the tables do not move)."""

    def __init__(self, model: Layer, loss_fn, lr: float = 1e-3, embed_l2: float = 0.0,
                 cuda_graph: bool = False, metrics=None):
        from .core import DenseAdam, StepGraph
        self._DenseAdam = DenseAdam
        self.model, self.loss_fn, self.lr = model, loss_fn, lr
        self.metrics = list(metrics or [])
        self.cuda_graph = cuda_graph
        self._evaluator = None
        self.tables = [m for m in model.modules() if isinstance(m, EmbeddingTables)]
        for ts in self.tables:
            if ts.optimizer is None:
                ts.set_optimizer(SparseOptimizer("adam", lr=lr, l2=embed_l2))
        self.dense_opt = None
        # cuda_graph: replay the step from a CUDA graph (core.StepGraph) — for the launch-bound
        # small models; per-step host values (the Adam step size, YoutubeDNN's sampler seed)
        # move to device scalars refreshed before each replay
        self.graph = StepGraph(self._body, self._advance) if cuda_graph else None

    def _setup(self, inputs):
        was = self.model.training
        self.model.eval()
        with torch.no_grad():
            self.model(inputs)
        self.model.train(was)
        emb = {id(p) for ts in self.tables for p in ts.parameters()}
        params = [p for p in self.model.parameters() if id(p) not in emb and p.requires_grad]
        self.dense_opt = self._DenseAdam(params, lr=self.lr)
        if self.graph is not None:
            self.dense_opt.enable_device_lr()
            for ts in self.tables:
                if ts.optimizer is not None:
                    ts.optimizer.enable_device_lr(self.dense_opt.flat.device)
            if hasattr(self.model, "enable_device_seed"):       # per-step host values -> memory
                self.model.enable_device_seed(self.dense_opt.flat.device)

    def _advance(self):
        seen = set()
        for ts in self.tables:          # one optimizer object may serve several table sets
            if ts.optimizer is not None and id(ts.optimizer) not in seen:
                seen.add(id(ts.optimizer))
                ts.begin_step()
        self.dense_opt.advance()
        if getattr(self.model, "seed_dev", None) is not None:
            self.model.advance()

    def _body(self, inputs, labels):
        out = self.model(inputs)
        loss = self.loss_fn(out, labels)
        for m in self.metrics:
            m.update_state(labels, out.detach())
        self.dense_opt.zero_grad()
        loss.backward()
        self.dense_opt.apply()
        for ts in self.tables:
            ts.wait_pending()
        return loss.detach()

    def step(self, inputs, labels=None) -> torch.Tensor:
        if self.dense_opt is None:
            self._setup(inputs)
        if self.graph is not None:
            return self.graph(inputs, labels)
        self._advance()
        return self._body(inputs, labels)

    def _eval_forward(self, inputs, labels):
        out = self.model(inputs)
        return out, self.loss_fn(out, labels)

    def evaluate(self, batches) -> dict:
        """Keras `model.evaluate` over `(inputs, labels)` pairs: the mean loss (weighted by batch
        size) and every metric of the trainer, computed by fresh copies of the metrics.  Changes
        no parameter, buffer, table, optimizer state or step counter (metrics.Evaluator)."""
        if isinstance(self.model, YoutubeDNN):
            raise TypeError("Trainer.evaluate: YoutubeDNN's forward advances its sampler seed; "
                            "matching models are not evaluated here")
        if self._evaluator is None:
            from .metrics import Evaluator
            self._evaluator = Evaluator(self._eval_forward, self.metrics, self.cuda_graph)

        def prepare(inputs):
            if self.dense_opt is None:      # build the layers and flatten before any capture
                self._setup(inputs)
        return self._evaluator.run(self.model, batches, prepare)
