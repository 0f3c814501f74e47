"""metrics.AUC on the GPU (csrc/metrics.cu) against the oracle (SURVEY App. A19), and the trainers'
evaluate() / metrics= against hand-written loops."""
import numpy as np
import pytest
import torch

from oracle import metrics as O

pytestmark = pytest.mark.gpu

F32 = np.float32


def _preds(kind, n, T, rng):
    if kind == "uniform":
        return rng.random(n, dtype=F32)
    if kind == "clustered":      # a trained model near its base rate: two buckets
        lo, hi = 0.03, 0.04
        p = np.where(rng.random(n) < 0.7, lo, hi) + rng.random(n) * 1e-4
        return p.astype(F32)
    # thresholds k/(T-1) in fp32, their fp32 neighbours, 0.0 and 1.0
    t = (np.arange(T, dtype=F32) / F32(T - 1)).astype(F32)
    cand = np.concatenate([t, np.nextafter(t, F32(2)), np.nextafter(t, F32(-1)), [F32(0), F32(1)]])
    cand = cand[(cand >= 0) & (cand <= 1)]
    return rng.choice(cand, n).astype(F32)


@pytest.mark.parametrize("T", [2, 3, 200, 4096])
@pytest.mark.parametrize("kind", ["uniform", "clustered", "thresholds"])
def test_counts_bit_equal_to_oracle(rtf, T, kind):
    rng = np.random.default_rng(T * 7 + len(kind))
    for n in (0, 1, 31, 65536, 3_000_001):
        p = _preds(kind, n, T, rng)
        y = (rng.random(n) < 0.3).astype(F32).reshape(-1, 1)
        m = rtf.metrics.AUC(num_thresholds=T)
        m.build("cuda")
        m.update_state(torch.from_numpy(y).cuda(), torch.from_numpy(p).cuda().reshape(-1, 1))
        want, bad = O.auc_counts(y, p, T)
        assert not bad
        got = m.counts.cpu().numpy()
        assert np.array_equal(got, want), (n, np.abs(got - want).max())
        assert abs(float(m.result()) - O.auc_from_counts(want)) <= 1e-7
        m.check()


def test_keras_docstring_example(rtf):
    m = rtf.metrics.AUC(num_thresholds=3)
    m.update_state(torch.tensor([0, 0, 1, 1], device="cuda"), torch.tensor([0, 0.5, 0.3, 0.9], device="cuda"))
    assert m.counts.cpu().tolist() == [[1, 1, 0], [2, 0, 0]]
    assert float(m.result()) == 0.75


def test_slices_sum_to_one_update_and_reset_keeps_addresses(rtf):
    rng = np.random.default_rng(1)
    p = torch.from_numpy(rng.random(100_003, dtype=F32)).cuda()
    y = torch.from_numpy((rng.random(100_003) < 0.4).astype(F32)).cuda()
    whole, parts = rtf.metrics.AUC(), rtf.metrics.AUC()
    whole.update_state(y, p)
    for idx in torch.tensor_split(torch.arange(p.numel(), device="cuda"), 10):
        parts.update_state(y[idx], p[idx])
    assert torch.equal(whole.counts, parts.counts)
    assert torch.equal(whole.result(), parts.result())
    ptrs = (parts.counts.data_ptr(), parts.err.data_ptr())
    parts.reset_state()
    assert (parts.counts.data_ptr(), parts.err.data_ptr()) == ptrs
    assert int(parts.counts.sum()) == 0 and float(parts.result()) == 0.0


def test_invalid_input_raises_and_valid_elements_still_count(rtf):
    p = np.array([0.2, 1.5, 0.7, -0.1, np.nan, 0.4, 0.9, 1.0, 0.0], dtype=F32)
    y = np.array([1, 0, 0, 1, 1, 0.5, 1, 0, 1], dtype=F32)
    valid = [0, 2, 6, 7, 8]
    for sel in [valid + [b] for b in (1, 3, 4, 5)] + [list(range(len(p)))]:
        m = rtf.metrics.AUC()
        m.update_state(torch.from_numpy(y[sel]).cuda(), torch.from_numpy(p[sel]).cuda())
        want, flagged = O.auc_counts(y[sel], p[sel], 200)
        assert flagged and int(want.sum()) == len(valid)
        assert np.array_equal(m.counts.cpu().numpy(), want)
        with pytest.raises(ValueError):
            m.check()
        m.reset_state()
        m.check()


# ------------------------------------------------------------------------------------ trainers
ROWS = [50, 7, 1000, 33, 5000, 12]


def _ctr_batches(n, B, n_dense, rows, seed):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        dense = torch.rand(B, n_dense, generator=g)
        sparse = torch.stack([torch.randint(0, r, (B,), generator=g) for r in rows], 1).to(torch.int32)
        y = torch.randint(0, 2, (B, 1), generator=g).float()
        out.append(([dense.cuda(), sparse.cuda()], y.cuda()))
    return out


def _din_batches(n, B, seed, L=20):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        hist = torch.stack([torch.randint(1, 1000, (B, L), generator=g), torch.randint(1, 50, (B, L), generator=g)], -1)
        lens = torch.randint(1, L + 1, (B,), generator=g)
        hist[torch.arange(L)[None, :] >= lens[:, None]] = 0
        target = torch.stack([torch.randint(1, 1000, (B,), generator=g), torch.randint(1, 50, (B,), generator=g)], -1)
        y = torch.randint(0, 2, (B, 1), generator=g).float()
        out.append(([hist.to(torch.int32).cuda(), target.to(torch.int32).cuda()], y.cuda()))
    return out


def _fc(n_dense, rows, D):
    return [[{"feat": f"I{i}"} for i in range(n_dense)],
            [{"feat": f"C{i}", "feat_num": r, "embed_dim": D} for i, r in enumerate(rows)]]


DLRM_ROWS = [100, 5000, 17, 900, 100000, 3, 64, 2048]


def _make(rtf, name, graph=False, metrics=None):
    """-> (trainer, make_batches(n, B, seed) -> [(inputs, labels)], is_dlrm)"""
    torch.manual_seed(7)
    bce = lambda out, y: rtf.layers.binary_crossentropy(y, out)      # noqa: E731
    if name.startswith("dlrm"):
        m = rtf.DLRM(_fc(13, DLRM_ROWS, 16), bot_dnn_hidden_units=(32, 16), top_dnn_hidden_units=(64, 32),
                     interaction=name.split("_")[1], seed=1).cuda()
        tr = rtf.DLRMTrainer(m, lr=1e-2, cuda_graph=graph, metrics=metrics)
        return tr, lambda n, B, s: _ctr_batches(n, B, 13, DLRM_ROWS, s), True
    if name == "fm":
        m = rtf.FMModel(_fc(4, ROWS, 8), k=8, seed=3)
    elif name == "deepfm":
        m = rtf.models.DeepFM(_fc(4, ROWS, 8), hidden_units=(32, 16), seed=3)
    elif name == "autoint":
        m = rtf.models.AutoInt(_fc(4, ROWS, 16), head_size=16, head_num=2, n_layers=2, seed=3)
    elif name == "din":
        m = rtf.models.DIN([1000, 50], embed_dim=8, maxlen=20, seed=3)
        tr = rtf.models.Trainer(m, bce, lr=1e-2, cuda_graph=graph, metrics=metrics)
        return tr, lambda n, B, s: _din_batches(n, B, s), False
    tr = rtf.models.Trainer(m, bce, lr=1e-2, cuda_graph=graph, metrics=metrics)
    return tr, lambda n, B, s: _ctr_batches(n, B, 4, ROWS, s), False


def _train(tr, batches, dlrm):
    for inputs, y in batches:
        tr.step(*inputs, y) if dlrm else tr.step(inputs, y)


def _eval(tr, batches, dlrm):
    return tr.evaluate([(x[0], x[1], y) for x, y in batches] if dlrm else batches)


def _state(tr):
    """Every parameter, buffer, table, optimizer moment and step counter of a trainer's model."""
    m = tr.model
    s = {f"p.{k}": v.detach().clone() for k, v in m.named_parameters()}
    s.update({f"b.{k}": v.detach().clone() for k, v in m.named_buffers()})
    tsets = [t for t in m.modules() if hasattr(t, "state1")]          # EmbeddingTables
    for i, ts in enumerate(tsets):
        for j, t in enumerate(ts.state1 + ts.state2):
            if t is not None:
                s[f"opt.{i}.{j}"] = t.clone()
        s[f"step.{i}"] = ts.optimizer.step
    for k in ("flat", "flat_grad", "m", "v"):
        s[f"dense.{k}"] = getattr(tr.dense_opt, k).clone()
    s["dense.t"] = tr.dense_opt.t
    return s


def _assert_same_state(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if isinstance(a[k], torch.Tensor):
            assert torch.equal(a[k], b[k]), k
        else:
            assert a[k] == b[k], k


def _bce64(y, p):
    p = np.clip(p.astype(np.float64), 1e-7, float(F32(1 - 1e-7)))
    return float(-np.mean(y * np.log(p + 1e-7) + (1 - y) * np.log(1 - p + 1e-7)))


@pytest.mark.parametrize("name", ["fm", "deepfm", "autoint", "din", "dlrm_dot", "dlrm_cat"])
def test_evaluate_matches_a_hand_written_loop(rtf, name):
    tr, make, dlrm = _make(rtf, name, metrics=[rtf.metrics.AUC()])
    _train(tr, make(4, 512, 1), dlrm)
    assert tr.model.training
    ev = make(3, 512, 2) + make(1, 200, 3)
    before = _state(tr)
    train_counts = tr.metrics[0].counts.clone()
    got = _eval(tr, ev, dlrm)
    assert tr.model.training
    _assert_same_state(before, _state(tr))
    assert torch.equal(train_counts, tr.metrics[0].counts)      # training-time metric untouched

    tr.model.eval()
    preds, losses, sizes = [], [], []
    with torch.no_grad():
        for x, y in ev:
            p = tr.model(x).cpu().numpy().reshape(-1)
            yy = y.cpu().numpy().reshape(-1)
            preds.append((yy, p))
            losses.append(_bce64(yy, p))
            sizes.append(len(yy))
    tr.model.train()
    y_all = np.concatenate([a for a, _ in preds])
    p_all = np.concatenate([b for _, b in preds])
    counts, bad = O.auc_counts(y_all, p_all, 200)
    assert not bad
    assert np.array_equal(tr._evaluator.metrics[0].counts.cpu().numpy(), counts)
    assert set(got) == {"loss", "auc"}
    assert abs(got["auc"] - O.auc_from_counts(counts)) <= 1e-7
    want_loss = float(np.dot(losses, sizes) / sum(sizes))
    assert abs(got["loss"] - want_loss) <= 1e-6 * abs(want_loss)


@pytest.mark.parametrize("name", ["deepfm", "dlrm_dot"])
def test_graph_evaluate_equals_eager_bitwise(rtf, name):
    runs = []
    for graph in (False, True):
        tr, make, dlrm = _make(rtf, name, graph=graph, metrics=[rtf.metrics.AUC()])
        _train(tr, make(5, 256, 1), dlrm)
        ev = make(6, 256, 2) + make(1, 100, 3)          # a ragged last batch runs eagerly
        r1 = _eval(tr, ev, dlrm)
        _train(tr, make(3, 256, 4), dlrm)
        r2 = _eval(tr, ev, dlrm)
        runs.append((r1, r2, tr))
    assert runs[1][2]._evaluator.graph.n_replays == 3 + 6
    assert runs[0][0] == runs[1][0] and runs[0][1] == runs[1][1]
    assert runs[0][0] != runs[0][1]


@pytest.mark.parametrize("name", ["fm", "dlrm_dot"])
def test_metrics_during_training(rtf, name):
    trs = []
    for graph, metrics in ((False, True), (True, True), (False, False)):
        tr, make, dlrm = _make(rtf, name, graph=graph, metrics=[rtf.metrics.AUC()] if metrics else None)
        bs = make(7, 256, 1)
        _train(tr, bs, dlrm)
        trs.append(tr)
    eager, graph, plain = trs
    assert graph.graph.n_replays == 4
    assert torch.equal(eager.metrics[0].counts, graph.metrics[0].counts)
    assert int(eager.metrics[0].counts.sum()) == 7 * 256
    assert torch.equal(eager.metrics[0].result(), graph.metrics[0].result())
    eager.metrics[0].check()
    for tr in (eager, graph):
        _assert_same_state(_state(plain), _state(tr))


def test_no_grad_dlrm_forward_launches_no_embedding_backward(rtf):
    from torch.profiler import ProfilerActivity, profile
    tr, make, _ = _make(rtf, "dlrm_dot", metrics=[rtf.metrics.AUC()])
    (x, y), = make(1, 1024, 1)
    tr.evaluate([(x[0], x[1], y)])                      # layers built, kernels loaded
    torch.cuda.synchronize()
    k2 = ("make_keys", "sort_hist", "sort_scatter", "scan_tile", "seg_apply")

    def kernels(fn):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return [e.name for e in prof.events() if e.device_type.name == "CUDA"]

    names = kernels(lambda: tr.evaluate([(x[0], x[1], y)]))
    assert any("dot_fwd" in n for n in names) and any("auc_update" in n for n in names)
    assert not [n for n in names if any(k in n for k in k2)]
    names = kernels(lambda: tr.step(x[0], x[1], y))    # the training step still prepares K2
    assert all(any(k in n for n in names) for k in ("make_keys", "seg_apply"))


def test_evaluate_refuses_a_model_whose_forward_has_side_effects(rtf):
    m = rtf.models.YoutubeDNN([100, 50], item_num=500, embed_dim=8, user_dnn_hidden_units=(16, 8),
                              num_sampled=8, seed=4)
    tr = rtf.models.Trainer(m, lambda out, y: out.mean(), metrics=[rtf.metrics.AUC()])
    with pytest.raises(TypeError):
        tr.evaluate([([torch.zeros(4, 2, dtype=torch.int32, device="cuda"),
                       torch.zeros(4, dtype=torch.int64, device="cuda")], None)])
    assert m._step == 0
