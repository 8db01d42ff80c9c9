"""Layer / model tests (reference tests/test_layers.py strategy + arena checks)."""
import os

import numpy as np
import pytest
import torch

from shallowspeed_b200.layers import MLP, Linear, MSELoss, ParamArena, Sequential, Softmax
from shallowspeed_b200.models.layers import param_ld
from shallowspeed_b200.optimizer import SGD


def test_sequential_forward_backward_zero_grad():
    layers = [Linear(12, 8), Linear(8, 6), Linear(6, 4, activation=None), Softmax()]
    model = Sequential(layers)
    assert len(model.parameters()) == 6
    x = torch.randn(5, 12)
    out = model(x)
    assert out.shape == (5, 4) and out.dtype == torch.float32
    assert torch.allclose(out.sum(dim=1), torch.ones(5), atol=1e-5)
    model.backward(torch.randn(5, 4))
    for p in model.parameters():
        assert p.grad.shape == p.data.shape
    assert any(float(p.grad.abs().sum()) > 0 for p in model.parameters())
    model.zero_grad()
    for p in model.parameters():
        assert float(p.grad.abs().sum()) == 0.0


def test_mlp_partitioner():
    sizes = [13, 12, 11, 10, 9, 8, 7, 6, 5]
    first = MLP(sizes, 0, 3, batch_size=4)
    assert first.in_dim == 13 and first.out_dim == 10 and len(first.layers) == 3
    assert all(l.activation is not None for l in first.layers)
    last = MLP(sizes, 2, 3, batch_size=4)
    assert last.in_dim == 7 and last.out_dim == 5
    assert len(last.layers) == 4  # 2 Linear + Softmax + MSELoss
    assert last.layers[0].activation is not None and last.layers[1].activation is None
    assert isinstance(last.layers[-1], MSELoss) and isinstance(last.layers[-2], Softmax)
    with pytest.raises(AssertionError):
        MLP(sizes, 0, 2, batch_size=4)


def test_default_model_partition_param_counts():
    sizes = [784, 128, 127, 126, 125, 124, 123, 10]
    count = lambda m: sum(p.data.numel() for p in m.parameters())
    assert count(MLP(sizes, 0, 1, 128)) == 181105
    assert [count(MLP(sizes, s, 2, 128)) for s in range(2)] == [148866, 32239]
    assert [count(MLP(sizes, s, 4, 128)) for s in range(4)] == [116863, 32003, 30999, 1240]
    m7 = MLP(sizes, 7, 8, 128)   # reference quirk: pp=8 last stage is Softmax+MSE only
    assert count(m7) == 0 and m7.in_dim == 10 and m7.out_dim == 10
    assert MLP(sizes, 6, 8, 128).layers[0].activation is not None


def test_init_is_layout_independent_and_matches_reference_recipe():
    from numpy.random import MT19937, RandomState, SeedSequence

    sizes = [784, 128, 127, 126, 125, 124, 123, 10]
    full = MLP(sizes, 0, 1, 128)
    parts = [MLP(sizes, s, 4, 128) for s in range(4)]
    flat = [p for m in parts for p in m.parameters()]
    for a, b in zip(full.parameters(), flat):
        assert torch.equal(a.data, b.data)
    rs = RandomState(MT19937(SeedSequence(784 + 128 * 1337)))
    w = rs.normal(0.0, 1.0, (128, 784)).astype(np.float32) / np.float32(np.sqrt(784))
    assert np.array_equal(full.parameters()[0].data.numpy(), w.astype(np.float32))
    assert full.parameters()[0].data.dtype == torch.float32


def test_arena_layout_and_views():
    arena = ParamArena([(128, 784), (127, 128), (10, 123)])
    for i, (o, k) in enumerate(arena.blocks):
        assert arena.lds[i] == param_ld(k) and arena.lds[i] % 8 == 0 and arena.lds[i] >= k + 1
        assert arena.offsets[i] % 32 == 0          # 128-byte aligned block base (TMA)
        assert arena.weight_view(i).shape == (o, k)
        assert arena.bias_view(i).shape == (1, o)
    arena.weight_view(1).fill_(2.0)
    arena.bias_view(1).fill_(3.0)
    blk = arena.block(1)
    assert float(blk[:, :128].min()) == 2.0 and float(blk[:, 128].min()) == 3.0
    assert float(blk[:, 129:].abs().sum()) == 0.0
    assert float(arena.block(0).abs().sum()) == 0.0


def test_fused_arena_sgd_equals_per_param_sgd():
    sizes = [20, 16, 12, 10]
    a, b = MLP(sizes, 0, 1, 8), MLP(sizes, 0, 1, 8)
    x, t = torch.randn(8, 20), torch.eye(10)[:8]
    for m in (a, b):
        m.forward(x)
        m.backward(t)
    SGD(a.parameters(), 0.1, arena=a.arena).step()
    SGD(b.parameters(), 0.1).step()
    for p, q in zip(a.parameters(), b.parameters()):
        assert torch.allclose(p.data, q.data, atol=1e-7)


def test_microbatch_accumulation_equals_full_batch():
    sizes = [784, 128, 127, 126, 125, 124, 123, 10]
    x = torch.randn(32, 784)
    t = torch.eye(10)[torch.randint(0, 10, (32,))]
    full, acc = MLP(sizes, 0, 1, 32), MLP(sizes, 0, 1, 32)
    full.forward(x, 0)
    full.backward(t, 0)
    for mu in range(4):
        acc.forward(x[mu * 8:(mu + 1) * 8], mu)
    for mu in reversed(range(4)):
        acc.backward(t[mu * 8:(mu + 1) * 8], mu)
    for p, q in zip(full.parameters(), acc.parameters()):
        assert torch.allclose(p.grad, q.grad, atol=2e-6)


def test_matches_reference_model_numerics():
    """Same init, same forward, same gradients as the reference's NumPy model, element for element.  Its results are
    stored in tests/golden/reference_mlp_numerics.npz (oracle/make_golden.py): the output and biases in full, the
    weights as every row and column sum plus a seeded sample of elements, and each weight gradient as the two factors
    the reference multiplies (output gradient G and layer input A: dW = G.T @ A)."""
    from numpy.random import MT19937, RandomState, SeedSequence

    ref = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_mlp_numerics.npz"))
    sizes = [784, 128, 127, 126, 125, 124, 123, 10]
    ours = MLP(sizes, 0, 1, 128)
    rs = np.random.RandomState(0)
    x = rs.randn(32, 784).astype(np.float32)
    t = np.eye(10, dtype=np.float32)[rs.randint(0, 10, 32)]
    out = ours.forward(torch.from_numpy(x), 0)
    assert np.allclose(ref["out"], out.numpy(), atol=1e-5)
    ours.backward(torch.from_numpy(t), 0)
    params = ours.parameters()
    assert len(params) == 2 * (len(sizes) - 1)
    for i, (w, b) in enumerate(zip(params[0::2], params[1::2])):
        n_out, n_in = w.data.shape
        # the reference's init recipe as it runs under NumPy >= 2: fp32 normals divided in fp64 (SURVEY.md fact 5);
        # it reproduces the stored sample exactly and every row and column sum to rounding, i.e. every element
        w_ref = RandomState(MT19937(SeedSequence(n_in + n_out * 1337))).normal(0.0, 1.0, (n_out, n_in)).astype(np.float32)
        w_ref = (w_ref.astype(np.float64) / np.sqrt(n_in)).astype(np.float32)
        assert np.array_equal(ref[f"W{i}_sample"], w_ref.reshape(-1)[ref[f"W{i}_idx"]])
        assert np.allclose(ref[f"W{i}_rowsum"], w_ref.astype(np.float64).sum(axis=1), atol=1e-12, rtol=0)
        assert np.allclose(ref[f"W{i}_colsum"], w_ref.astype(np.float64).sum(axis=0), atol=1e-12, rtol=0)
        # the intended fp32 values agree to 1 ulp
        assert np.allclose(w_ref, w.data.numpy(), atol=1e-7, rtol=0)
        assert np.allclose(ref[f"b{i}"], b.data.numpy(), atol=1e-7, rtol=0)
        a = ref[f"A{i}"] if i else x
        dw_ref = ref[f"G{i}"].astype(np.float64).T @ a.astype(np.float64)
        assert np.allclose(dw_ref, w.grad.numpy(), atol=1e-5)
        assert np.allclose(ref[f"db{i}"], b.grad.numpy(), atol=1e-5)
