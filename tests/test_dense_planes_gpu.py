"""Plane-fed dense GEMM (csrc/dense_gemm_planes.cuh): the device split equals its numpy
restatement bit for bit, and the GEMM fed those planes equals the fp32-fed GEMM bit for bit —
at every shape the DLRM bench step runs, in all three layouts, and on ragged tails."""
import numpy as np
import pytest
import torch

from test_dense_planes_cpu import bf16_bits, edge_values, split_ref

pytestmark = pytest.mark.gpu

from recommend_tf2_b200 import core  # noqa: E402

M_BENCH = 65536
# (K_in, N_out) of the DLRM bench MLP layers the tensor-core GEMM runs: top 480-1024-1024-512-256,
# bottom 512-256-128 (the 13-wide input and the 1-wide output layer take other paths)
BENCH_LAYERS = [(480, 1024), (1024, 1024), (1024, 512), (512, 256), (512, 256), (256, 128)]
BENCH_LAYERS = sorted(set(BENCH_LAYERS))


def _planes(x):
    return core.split_planes(x.contiguous())


def test_device_split_matches_restatement(rtf):
    x = edge_values(np.random.default_rng(2))
    x = np.concatenate([x, np.array([np.inf, -np.inf], np.float32)])
    # (2, 4k): the flat vectorized pass; (k, 6): the per-pair pass for rows that are not quads
    for x2 in (x[: x.size // 8 * 8].reshape(2, -1), x[: x.size // 6 * 6].reshape(-1, 6)):
        got = _planes(torch.from_numpy(x2).cuda()).view(torch.int16).cpu().numpy().view(np.uint16)
        for p, want in enumerate(split_ref(x2)):
            assert np.array_equal(got[p], bf16_bits(want)), f"plane {p}, shape {x2.shape}"


def test_split_pads_nothing_and_keeps_row_order(rtf):
    x = torch.randn(37, 10, device="cuda")
    p = _planes(x).float()
    back = p[0].double() + p[1].double() * 2.0 ** -8 + p[2].double() * 2.0 ** -16
    assert torch.allclose(back, x.double(), rtol=2.0 ** -23, atol=0)


def _gemm_pair(kind, a, b, bias=None, relu=False, splits=1):
    want = core.dense_gemm(kind, a, b, bias, relu, splits=splits)
    got = core.dense_gemm_planes(kind, _planes(a), _planes(b), bias, relu, splits=splits)
    return got, want


@pytest.mark.parametrize("K,N", BENCH_LAYERS)
@pytest.mark.parametrize("relu", [False, True])
def test_nn_bench_shapes_bit_identical(rtf, K, N, relu):
    x = torch.randn(M_BENCH, K, device="cuda")
    w = torch.randn(K, N, device="cuda") * K ** -0.5
    b = torch.randn(N, device="cuda")
    got, want = _gemm_pair("nn", x, w, b, relu)
    assert torch.equal(got, want)


@pytest.mark.parametrize("K,N", BENCH_LAYERS)
def test_nt_bench_shapes_bit_identical(rtf, K, N):
    g = torch.randn(M_BENCH, N, device="cuda")
    w = torch.randn(K, N, device="cuda") * K ** -0.5
    got, want = _gemm_pair("nt", g, w)
    assert torch.equal(got, want)


@pytest.mark.parametrize("K,N", BENCH_LAYERS)
def test_tn_bench_shapes_split_k_bit_identical(rtf, K, N):
    x = torch.relu(torch.randn(M_BENCH, K, device="cuda"))
    g = torch.randn(M_BENCH, N, device="cuda") * 1e-3
    splits = core._wgrad_splits(M_BENCH, K, N)
    got, want = _gemm_pair("tn", x, g, splits=splits)
    assert torch.equal(got, want)
    got1, want1 = _gemm_pair("tn", x[:4096], g[:4096])
    assert torch.equal(got1, want1)


@pytest.mark.parametrize("M,K,N", [(1000, 40, 72), (300, 264, 136), (257, 8, 8), (5000, 1032, 392)])
def test_ragged_tails_bit_identical(rtf, M, K, N):
    """M, N and K that are not multiples of the 256 x 128 x 32 tile, bias and ReLU on and off"""
    a = torch.randn(M, K, device="cuda")
    w = torch.randn(K, N, device="cuda")
    b = torch.randn(N, device="cuda")
    for bias, relu in ((None, False), (b, True)):
        got, want = _gemm_pair("nn", a, w, bias, relu)
        assert torch.equal(got, want)
    got, want = _gemm_pair("nt", torch.randn(M, N, device="cuda"), w)
    assert torch.equal(got, want)
    got, want = _gemm_pair("tn", a, torch.randn(M, N, device="cuda"))
    assert torch.equal(got, want)


def test_wide_dynamic_range_bit_identical(rtf):
    x = torch.randn(4096, 256, device="cuda") * torch.exp2(
        torch.randint(-20, 21, (4096, 256), device="cuda").float())
    w = torch.randn(256, 128, device="cuda")
    got, want = _gemm_pair("nn", x, w)
    assert torch.equal(got, want)


def test_plane_gemm_rejects_misaligned_planes(rtf):
    a = torch.zeros(3, 64, 12, dtype=torch.bfloat16, device="cuda")   # K = 12: rows not 16 B
    w = torch.zeros(3, 12, 64, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(Exception):
        core.dense_gemm_planes("nn", a, w)


def test_dense_layers_planes_vs_fp32_path_bit_identical(rtf):
    """Two Dense layers at DLRM top-MLP widths (480 -> 1024 -> 1024, ReLU), forward and backward:
    the plane-fed path (the default for these widths) equals the fp32-fed path bit for bit."""
    assert core._planes_pay(4096, 480, 1024) and core._planes_pay(4096, 1024, 1024)
    x0 = torch.randn(4096, 480, device="cuda")
    res = {}
    for planes in (True, False):
        core.set_dense_planes(planes)
        torch.manual_seed(0)
        l1, l2 = core.Dense(1024, activation="relu"), core.Dense(1024, activation="relu")
        x = x0.clone().requires_grad_(True)
        y = l2(l1(x))
        (y * torch.linspace(-1, 1, 1024, device="cuda")).sum().backward()
        res[planes] = [y.detach(), x.grad, l1.kernel.grad, l1.bias.grad, l2.kernel.grad, l2.bias.grad]
    core.set_dense_planes(True)
    for a, b in zip(res[True], res[False]):
        assert torch.equal(a, b)


def _dlrm_batches(rows, n, B, seed=0):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        dense = torch.rand(B, 13, generator=g)
        sparse = torch.stack([torch.randint(0, r, (B,), generator=g) for r in rows], 1).to(torch.int32)
        y = torch.randint(0, 2, (B, 1), generator=g).float()
        out.append((dense.cuda(), sparse.cuda(), y.cuda()))
    return out


@pytest.mark.parametrize("pad_to", [1, 8])
@pytest.mark.parametrize("graph", [False, True])
def test_dlrm_training_planes_vs_fp32_path_bit_identical(rtf, pad_to, graph):
    """N DLRM training steps at the bench's interaction width (26 tables, D = 128: 479 columns,
    zero-padded to 480 inside the layer for pad_to=1, 480 from the interaction for pad_to=8) and
    top-MLP widths that take the plane path: loss, dense parameters and table rows are
    bit-identical with planes and with the fp32-fed GEMM forced, eager and graph-replayed."""
    F, D, B, steps = 26, 128, 2048, 6
    rows = [97 + 31 * i for i in range(F)]
    fc = [[{"feat": f"I{i}"} for i in range(13)],
          [{"feat": f"C{i}", "feat_num": rows[i], "embed_dim": D} for i in range(F)]]
    assert rtf.dot_out_cols(F + 1, D, pad_to) == (479 if pad_to == 1 else 480)
    assert core._planes_pay(B, 480, 1024) and core._planes_pay(B, 1024, 512)
    bs = _dlrm_batches(rows, steps, B)
    runs = {}
    try:
        for planes in (True, False):
            core.set_dense_planes(planes)
            torch.manual_seed(5)
            m = rtf.DLRM(fc, bot_dnn_hidden_units=(64, D), top_dnn_hidden_units=(1024, 512, 64),
                         seed=1, pad_to=pad_to).cuda()
            tr = rtf.DLRMTrainer(m, lr=1e-3, cuda_graph=graph)
            losses = [float(tr.step(d, s, y)) for d, s, y in bs]
            runs[planes] = (losses, tr.dense_opt.flat.clone(),
                            [w.detach().clone() for w in m.embed_layers.weights])
            if graph:
                assert tr.graph.n_replays > 0
    finally:
        core.set_dense_planes(True)
    (l1, p1, t1), (l0, p0, t0) = runs[True], runs[False]
    assert l1 == l0
    assert torch.equal(p1, p0)
    for a, b in zip(t1, t0):
        assert torch.equal(a, b)


@pytest.mark.parametrize("width", [479, 1005])
def test_dense_layer_padded_input_width_takes_planes(rtf, width):
    """An input width that is not a multiple of 4 is zero-padded inside the layer; with N = 1024
    the padded layer takes the plane path and its gradients are sliced back to the input width."""
    x0 = torch.randn(2048, width, device="cuda")
    res = {}
    try:
        for planes in (True, False):
            core.set_dense_planes(planes)
            torch.manual_seed(0)
            layer = core.Dense(1024, activation="relu")
            x = x0.clone().requires_grad_(True)
            y = layer(x)
            (y * torch.linspace(-1, 1, 1024, device="cuda")).sum().backward()
            assert x.grad.shape == x0.shape and layer.kernel.grad.shape == (width, 1024)
            res[planes] = [y.detach(), x.grad, layer.kernel.grad, layer.bias.grad]
    finally:
        core.set_dense_planes(True)
    for a, b in zip(res[True], res[False]):
        assert torch.equal(a, b)
