"""CPU: sparse GPFQ (`l1_penalty`) -- the shrink, its closed form, the C and NumPy walks, argument validation and the mirror classes
on the sparse oracle engine.  The GPU tests (test_gpu_sparse.py) hold the CUDA path to the same oracle."""
import os

import numpy as np
import pytest

from conftest import glorot, golden, hidden_pair
from oracle import gpfq_oracle as O, sparse_oracle as SP, stochastic_oracle as SO
from quantized_neural_networks_b200 import QuantizedCNN, QuantizedNeuralNetwork
from test_host_channel_alphabets import QUIET, _cnn_data, _free_port, _mlp_data, channel_cnn, mlp


def with_sparse_oracle(cls, *args, **kw):
    q = cls(*args, **kw)
    q.__class__ = type("SparseOracle" + cls.__name__, (cls,), {"engine": property(lambda self: SP.SparseOracleEngine())})
    return q


def _weights_equal(a, b):
    for la, lb in zip(a.layers, b.layers):
        for wa, wb in zip(la.get_weights(), lb.get_weights()):
            if not np.array_equal(wa, wb):
                return False
    return True


def test_shrink_edge_cases():
    c = SP.lib().sp_shrink
    cases = [(0.0, 0.0, 0.0), (-0.0, 0.0, 0.0), (1.5, 0.5, 1.0), (-1.5, 0.5, -1.0), (0.5, 0.5, 0.0), (-0.5, 0.5, 0.0),
             (np.inf, 1.0, np.inf), (-np.inf, 1.0, -np.inf), (3.0, np.inf, 0.0), (np.inf, np.inf, 0.0), (1e-300, 0.0, 1e-300)]
    for v, tau, want in cases:
        got = float(SP.shrink(v, tau))
        assert got == want and np.signbit(got) == np.signbit(want), (v, tau, got)
        assert c(v, tau) == want, (v, tau)
    assert np.isnan(SP.shrink(np.nan, 0.5)) and np.isnan(c(np.nan, 0.5))
    # tau = +0 is the identity up to the sign of a zero
    v = np.random.default_rng(0).standard_normal(1000)
    assert np.array_equal(SP.shrink(v, 0.0), v)
    assert not np.signbit(SP.shrink(-0.0, 0.0))


def test_shrink_is_the_minimiser_of_the_one_step_problem():
    """argmin_p 1/2 (num - p den)^2 / den + lambda |p| (the one-step L1 problem along Xq_t, in the Gram form) is s_lambda(num) / den."""
    from scipy.optimize import minimize_scalar
    rng = np.random.default_rng(1)
    for _ in range(200):
        num, den, lam = rng.normal() * 10, rng.uniform(0.1, 20), rng.uniform(0, 15)
        f = lambda p: 0.5 * (num - p * den) ** 2 / den + lam * abs(p)
        closed = float(SP.step_value(num, den, lam))
        want = np.sign(num) * max(abs(num) - lam, 0.0) / den
        assert abs(closed - want) <= 1e-12 * (1 + abs(want))
        best = minimize_scalar(f, bounds=(-abs(num) / den - 1, abs(num) / den + 1), method="bounded",
                               options={"xatol": 1e-12}).x
        assert abs(best - closed) <= 1e-6 * (1 + abs(closed)), (num, den, lam)
        assert f(closed) <= f(best) + 1e-12


@pytest.mark.parametrize("name", ["dense_first_ternary", "dense_hidden_grid", "ties_and_dead"])
def test_zero_penalty_reproduces_the_oracles_on_golden_inputs(name):
    g = golden(name)
    keys = list(g.keys())
    X = g["X"].astype(np.float32)
    Xq = g["Xq"].astype(np.float32) if "Xq" in keys else X
    W = g["W"].astype(np.float32)
    akeys = [k for k in keys if k.startswith("A")] or []
    As = [g[k] for k in akeys] if akeys else [O.layer_alphabet(W, 2, O.unit_alphabet(np.log2(3)))]
    for A in As[:2]:
        A = np.asarray(A, np.float64)
        cols = list(range(min(W.shape[1], 6)))
        want = np.stack([O.quantize_neuron(W[:, j], X, Xq, A) for j in cols], axis=1)
        assert np.array_equal(SP.numpy_dense_layer(W[:, cols], X, Xq, A, 0.0), want), name
        assert np.array_equal(SP.dense_layer(W[:, cols], X, Xq, A, 0.0), want), name
        assert np.array_equal(SP.dense_layer(W, X, Xq, A, 0.0, seed=9), SO.dense_layer(W, X, Xq, A, 9)), name


@pytest.mark.parametrize("K", [3, 4, 5, 16])
def test_c_and_numpy_walks_are_equal(K):
    rng = np.random.default_rng(K)
    N0, N1, m = 40, 9, 120
    X, Xq = hidden_pair(rng, N0, m)
    X[:2] = Xq[:2] = 0.0
    W = glorot(rng, N0, N1)
    W[:, 3] = 0.0
    A = float(np.median(np.abs(W))) * 2 * np.linspace(-1, 1, K)
    den = float(np.median(np.sum(Xq.astype(np.float64) ** 2, axis=1)))
    s = 10.0 ** rng.uniform(-1, 1, N1)
    s[5] = 0.0
    for lam in (0.0, 0.3 * A[-1] * den, 1e300):
        for seed, scales in ((None, None), (7, None), (None, s), (7, s)):
            c = SP.dense_layer(W, X, Xq, A, lam, seed, scales)
            n = SP.numpy_dense_layer(W, X, Xq, A, lam, seed, scales)
            assert np.array_equal(c, n), (K, lam, seed, scales is None)
    if K % 2:
        assert not SP.dense_layer(W, X, Xq, A, 1e300).any()
        assert np.mean(SP.dense_layer(W, X, Xq, A, 0.3 * A[-1] * den) == 0) > np.mean(SP.dense_layer(W, X, Xq, A, 0.0) == 0)


def test_engine_penalty_arguments():
    from quantized_neural_networks_b200.engine import _l1_args
    assert _l1_args(None, 3) is None
    assert _l1_args(0.5, 2) == [0.5, 0.5] and _l1_args(0, 1) == [0.0]
    assert _l1_args([1, 2.5], 2) == [1.0, 2.5] and _l1_args(np.array([0.0, 3.0]), 2) == [0.0, 3.0]
    for bad, n in (([1.0], 2), (-1.0, 1), (np.inf, 1), (np.nan, 1), ("1", 1), (True, 1), ([None], 1), ({"a": 1}, 1)):
        with pytest.raises(ValueError):
            _l1_args(bad, n)


@pytest.mark.parametrize("bad", [-0.1, np.inf, np.nan, "0.5", True, {0: -1.0}, {"x": 1.0}, [0.5]])
def test_bad_penalties_raise(bad):
    with pytest.raises(ValueError):
        QuantizedNeuralNetwork(mlp(), 32, _mlp_data(), logger=QUIET, l1_penalty=bad)
    with pytest.raises(ValueError):
        QuantizedCNN(channel_cnn(), 8, _cnn_data(), logger=QUIET, l1_penalty=bad)


def test_penalty_needs_a_zero_level():
    with pytest.raises(ValueError, match="log2"):
        QuantizedNeuralNetwork(mlp(), 32, _mlp_data(), logger=QUIET, bits=2, l1_penalty=0.1)
    QuantizedNeuralNetwork(mlp(), 32, _mlp_data(), logger=QUIET, bits=np.log2(5), l1_penalty=0.1)
    QuantizedNeuralNetwork(mlp(), 32, _mlp_data(), logger=QUIET, bits=2)    # no penalty: any alphabet


def test_mirror_mlp_penalty_per_layer():
    net, seq = mlp(), _mlp_data()
    kw = dict(logger=QUIET, bits=np.log2(5), alphabet_scalar=3)
    q = with_sparse_oracle(QuantizedNeuralNetwork, net, 32, seq, l1_penalty={0: 2.0}, **kw)
    q.quantize_network()
    W = net.layers[0].get_weights()[0]
    X = np.asarray(seq.x, np.float32).T.copy()
    A = np.asarray(q._layer_alphabet(W), np.float64)
    assert np.array_equal(q.quantized_net.layers[0].get_weights()[0], SP.dense_layer(W, X, X, A, 2.0).astype(np.float32))
    plain = with_sparse_oracle(QuantizedNeuralNetwork, net, 32, seq, **kw)
    plain.quantize_network()
    zero = with_sparse_oracle(QuantizedNeuralNetwork, net, 32, seq, l1_penalty=0.0, **kw)
    zero.quantize_network()
    assert _weights_equal(plain.quantized_net, zero.quantized_net)
    W0 = q.quantized_net.layers[0].get_weights()[0]
    assert np.mean(W0 == 0) > np.mean(plain.quantized_net.layers[0].get_weights()[0] == 0)


@pytest.mark.parametrize("scope", ["layer", "channel"])
def test_mirror_cnn_conv_paths_agree(scope):
    net, seq = channel_cnn(), _cnn_data()
    kw = dict(logger=QUIET, bits=np.log2(3), alphabet_scalar=2, l1_penalty=0.5, alphabet_scope=scope)
    a = with_sparse_oracle(QuantizedCNN, net, 8, seq, conv_path="nhwc", **kw)
    b = with_sparse_oracle(QuantizedCNN, net, 8, seq, conv_path="patches", **kw)
    a.quantize_network()
    b.quantize_network()
    assert _weights_equal(a.quantized_net, b.quantized_net)
    c = with_sparse_oracle(QuantizedCNN, net, 8, seq, conv_path="nhwc", **dict(kw, l1_penalty=None))
    c.quantize_network()
    assert not _weights_equal(a.quantized_net, c.quantized_net)


def _shard_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        net, seq = channel_cnn(), _cnn_data()
        ok = True
        for path in ("nhwc", "patches"):
            kw = dict(logger=QUIET, bits=np.log2(3), alphabet_scalar=2, conv_path=path, l1_penalty={0: 0.5, 2: 1.0, 4: 0.25})
            one = with_sparse_oracle(QuantizedCNN, net, 8, seq, **kw)
            one.quantize_network()
            shr = with_sparse_oracle(QuantizedCNN, net, 8, seq, shard=(rank, world), **kw)
            shr.quantize_network()
            for idx in (0, 1, 2, 4):
                ok = ok and np.array_equal(one.quantized_net.layers[idx].get_weights()[0],
                                           shr.quantized_net.layers[idx].get_weights()[0])
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_shards_of_a_sparse_run_are_gathered(world):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_shard_worker, args=(r, world, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    assert dict(ret) == {r: True for r in range(world)}
