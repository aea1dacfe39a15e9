"""CPU: stochastic rounding (SPFQ, `rounding="stochastic"`) -- the draws, the quantizer, the C and NumPy walks, the layer seeds and
the mirror classes on the stochastic oracle engine.  The GPU tests (test_gpu_stochastic.py) hold the CUDA path to the same oracle."""
import os

import numpy as np
import pytest

from conftest import glorot, hidden_pair
from oracle import gpfq_oracle as O, stochastic_oracle as SO
from quantized_neural_networks_b200 import QuantizedCNN, QuantizedNeuralNetwork
from quantized_neural_networks_b200.quantized_network import layer_seed, splitmix64
from test_host_channel_alphabets import QUIET, _cnn_data, _free_port, _mlp_data, channel_cnn, mlp


def with_stochastic_oracle(cls, *args, **kw):
    q = cls(*args, **kw)
    q.__class__ = type("StochasticOracle" + cls.__name__, (cls,), {"engine": property(lambda self: SO.StochasticOracleEngine())})
    return q


def test_known_answers():
    assert splitmix64(0) == 0xE220A8397B1DCDAF
    assert splitmix64(0x9E3779B97F4A7C15) == 0x6E789E6AA1B965F4
    assert SO.splitmix64(0) == 0xE220A8397B1DCDAF and SO.lib().so_splitmix64(0) == 0xE220A8397B1DCDAF
    for seed, u, t, want in ((0, 0, 0, 0.13870941014555427), (1, 2, 3, 0.7684201926204703)):
        assert float(SO.draw(seed, u, t)) == want
        assert SO.lib().so_draw(seed, u, t) == want


def test_draws_are_exact_in_unit_interval_and_match_c():
    u = np.arange(5000)
    r = SO.draw(12345, u, 7)
    assert np.all((r >= 0) & (r < 1))
    assert np.all(r * 2.0 ** 53 == np.floor(r * 2.0 ** 53))
    c = np.array([SO.lib().so_draw(12345, int(x), 7) for x in u[:300]])
    assert np.array_equal(c, r[:300])


def _c_stoc_round(v, A, r):
    A = np.ascontiguousarray(A, dtype=np.float64)
    return SO.lib().so_stoc_round(float(v), A.ctypes.data, len(A), float(r))


def test_stoc_round_edge_cases():
    A = np.array([-1.0, -0.5, 0.0, 0.5, 1.0])
    cases = [(-1.0, 0.3, -1.0), (1.0, 0.3, 1.0), (-7.0, 0.9, -1.0), (7.0, 0.0, 1.0), (np.nan, 0.0, -1.0), (np.inf, 0.5, 1.0),
             (-np.inf, 0.5, -1.0), (0.5, 0.999, 0.5), (0.0, 0.0, 0.0), (0.25, 0.49, 0.5), (0.25, 0.5, 0.0), (-0.75, 0.0, -0.5)]
    for v, r, want in cases:
        got = SO.stoc_round(v, A, r)
        assert got == want, (v, r, got)
        assert _c_stoc_round(v, A, r) == want, (v, r)
    # duplicate levels: the interval is always the one above the last level <= v
    D = np.array([-1.0, 0.0, 0.0, 1.0])
    assert SO.stoc_round(0.0, D, 0.0) == 0.0 and SO.stoc_round(0.5, D, 0.49) == 1.0 and SO.stoc_round(0.5, D, 0.5) == 0.0
    assert SO.stoc_round(-0.5, D, 0.49) == 0.0 and SO.stoc_round(-0.5, D, 0.51) == -1.0
    assert _c_stoc_round(0.5, D, 0.49) == 1.0 and _c_stoc_round(-0.5, D, 0.51) == -1.0
    # a zero scale: every level is 0, so is every result
    Z = SO.unit_levels(A, 0.0)
    for v in (-3.0, -1e-300, 0.0, 2.0, np.nan):
        assert SO.stoc_round(v, Z, 0.3) == 0.0 and _c_stoc_round(v, Z, 0.3) == 0.0
    # one level
    assert SO.stoc_round(5.0, np.array([2.0]), 0.1) == 2.0 and _c_stoc_round(-5.0, np.array([2.0]), 0.1) == 2.0


@pytest.mark.parametrize("K", [3, 4, 16])
def test_stoc_round_is_unbiased(K):
    A = np.linspace(-1, 1, K)
    n = 200000
    r = SO.draw(99, np.arange(n), 0)
    for v in (-0.93, -0.31, 0.0, 0.123456, 0.77):
        q = SO.stoc_round(np.full(n, v), A, r)
        sigma = np.sqrt(max(np.var(q), 1e-30) / n)
        assert abs(q.mean() - v) <= 5 * sigma + 1e-15, (K, v, q.mean())
        lo = A[max(np.searchsorted(A, v, side="right") - 1, 0)]
        assert set(np.unique(q)) <= {lo, A[min(np.searchsorted(A, lo, side="right"), K - 1)]}


@pytest.mark.parametrize("bits", [np.log2(3), 2, 4])
def test_c_and_numpy_walks_are_equal(bits):
    rng = np.random.default_rng(int(bits * 10))
    N0, N1, m = 40, 9, 120
    X, Xq = hidden_pair(rng, N0, m)
    X[:2] = Xq[:2] = 0.0                        # dead directions
    W = glorot(rng, N0, N1)
    W[:, 3] = 0.0                               # a pruned neuron
    A = float(np.median(np.abs(W))) * 2 * O.unit_alphabet(bits)
    s = (10.0 ** rng.uniform(-1, 1, N1))
    s[5] = 0.0
    for scales in (None, s):
        for u0 in (0, 1000):
            c = SO.dense_layer(W, X, Xq, A, 77, scales, u0=u0)
            n = SO.numpy_dense_layer(W, X, Xq, A, 77, scales, u0=u0)
            assert np.array_equal(c, n), (bits, scales is None, u0)
    # shards see the global unit ids: a column range equals the same columns of the whole layer
    whole = SO.dense_layer(W, X, Xq, A, 5)
    part = SO.dense_layer(W, X, Xq, A, 5, j0=3, j1=7)
    assert np.array_equal(part[:, 3:7], whole[:, 3:7]) and not part[:, :3].any()
    # different seeds give different walks; the zero scale an all-zero column
    assert not np.array_equal(whole, SO.dense_layer(W, X, Xq, A, 6))
    assert not SO.dense_layer(W, X, Xq, A, 7, s)[:, 5].any()


def test_stochastic_walk_is_unbiased_on_a_single_step():
    """With one direction the walk rounds w alone: the mean over neurons (one draw each) is w."""
    rng = np.random.default_rng(1)
    N1 = 20000
    X = np.abs(rng.standard_normal((1, 30))).astype(np.float32)
    W = np.full((1, N1), 0.3, np.float32)
    A = O.unit_alphabet(2)
    Q = SO.dense_layer(W, X, X, A, 3)
    v = float(np.float32(0.3))
    sigma = np.sqrt(np.var(Q) / N1)
    assert abs(Q.mean() - v) < 5 * sigma


def test_layer_seed_derivation():
    assert layer_seed(0, 0) == splitmix64(splitmix64(0) ^ 0)
    assert layer_seed(7, 3) == splitmix64(splitmix64(7) ^ 3)
    assert len({layer_seed(s, i) for s in range(4) for i in range(6)}) == 24
    assert layer_seed(2 ** 64 - 1, 1) == splitmix64(splitmix64(2 ** 64 - 1) ^ 1)


@pytest.mark.parametrize("kw", [{"rounding": "floor"}, {"rounding": None}, {"rounding": "stochastic", "seed": -1},
                                {"rounding": "stochastic", "seed": 2 ** 64}, {"rounding": "stochastic", "seed": 1.5}])
def test_bad_rounding_arguments_raise(kw):
    with pytest.raises(ValueError):
        QuantizedNeuralNetwork(mlp(), 32, _mlp_data(), logger=QUIET, **kw)
    with pytest.raises(ValueError):
        QuantizedCNN(channel_cnn(), 8, _cnn_data(), logger=QUIET, **kw)


def test_engine_seed_arguments():
    from quantized_neural_networks_b200.engine import _seed_args
    assert _seed_args(None, 3) is None
    assert _seed_args(5, 3) == [5, 5, 5]
    assert _seed_args([1, 2], 2) == [1, 2] and _seed_args(np.array([1, 2], np.uint64), 2) == [1, 2]
    assert _seed_args(2 ** 64 - 1, 1) == [2 ** 64 - 1]
    for bad in ([1, 2], -1, 2 ** 64, 1.0, "3", True, [1.5], [None]):
        with pytest.raises(ValueError):
            _seed_args(bad, 1 if bad != [1, 2] else 3)


def _weights_equal(a, b):
    for la, lb in zip(a.layers, b.layers):
        for wa, wb in zip(la.get_weights(), lb.get_weights()):
            if not np.array_equal(wa, wb):
                return False
    return True


def test_mirror_mlp_walks_with_the_layer_seeds():
    net, seq = mlp(), _mlp_data()
    q = with_stochastic_oracle(QuantizedNeuralNetwork, net, 32, seq, logger=QUIET, bits=2, alphabet_scalar=3, rounding="stochastic",
                               seed=11)
    q.quantize_network()
    # layer 0 by hand: the C walk with layer_seed(11, 0)
    W = net.layers[0].get_weights()[0]
    X = np.asarray(seq.x, np.float32).T.copy()
    A = np.asarray(q._layer_alphabet(W), np.float64)
    assert np.array_equal(q.quantized_net.layers[0].get_weights()[0], SO.dense_layer(W, X, X, A, layer_seed(11, 0)).astype(np.float32))
    near = with_stochastic_oracle(QuantizedNeuralNetwork, net, 32, seq, logger=QUIET, bits=2, alphabet_scalar=3)
    near.quantize_network()
    assert not _weights_equal(q.quantized_net, near.quantized_net)
    again = with_stochastic_oracle(QuantizedNeuralNetwork, net, 32, seq, logger=QUIET, bits=2, alphabet_scalar=3,
                                   rounding="stochastic", seed=11)
    again.quantize_network()
    assert _weights_equal(q.quantized_net, again.quantized_net)


@pytest.mark.parametrize("scope", ["layer", "channel"])
def test_mirror_cnn_conv_paths_agree(scope):
    """Both conv paths of the mirror give the same stochastic weights: the patch path draws with the global unit ids."""
    net, seq = channel_cnn(), _cnn_data()
    kw = dict(logger=QUIET, bits=2, alphabet_scalar=3, rounding="stochastic", seed=5, alphabet_scope=scope)
    a = with_stochastic_oracle(QuantizedCNN, net, 8, seq, conv_path="nhwc", **kw)
    b = with_stochastic_oracle(QuantizedCNN, net, 8, seq, conv_path="patches", **kw)
    a.quantize_network()
    b.quantize_network()
    assert _weights_equal(a.quantized_net, b.quantized_net)
    c = with_stochastic_oracle(QuantizedCNN, net, 8, seq, conv_path="nhwc", **dict(kw, seed=6))
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
            kw = dict(logger=QUIET, bits=2, alphabet_scalar=3, conv_path=path, rounding="stochastic", seed=21)
            one = with_stochastic_oracle(QuantizedCNN, net, 8, seq, **kw)
            one.quantize_network()
            shr = with_stochastic_oracle(QuantizedCNN, net, 8, seq, shard=(rank, world), **kw)
            shr.quantize_network()
            for idx in (0, 1, 2, 4):
                ok = ok and np.array_equal(one.quantized_net.layers[idx].get_weights()[0],
                                           shr.quantized_net.layers[idx].get_weights()[0])
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_shards_of_a_stochastic_run_are_gathered(world):
    """Channel, group and neuron shards of a stochastic run, all-gathered under gloo, equal the one-rank run."""
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
