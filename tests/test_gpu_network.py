"""GPU: full-network parity through the reference-facing API (`QuantizedNeuralNetwork(...).quantize_network()`,
`QuantizedCNN(...).quantize_network()`, quantized_network.py:576-590 / :869-883).

The checker is the same host-side walk over the layers with the hot path replaced by the oracle (the C restatement of
`_quantize_neuron_parallel` / `_quantize_filter2D_parallel_jit`, pinned to the unmodified reference in test_oracle.py):
every layer sees the activations of the partially quantized network below it, exactly as in the reference.  Gates
(BASELINE.json north_star): per-layer agreement >= 99.99 %, relative residual within 1e-6, and IDENTICAL predictions /
accuracy of the quantized network on the synthetic evaluation set.
"""
import numpy as np
import pytest

from oracle import c_oracle, gpfq_oracle as O
from quantized_neural_networks_b200 import QuantizedCNN, QuantizedNeuralNetwork, hostnet

pytestmark = pytest.mark.gpu


class OracleEngine:
    """Test-only stand-in for GpfqEngine with the engine's call surface; routes the hot path through the oracle."""

    last_stats = {}

    def dense_layer(self, X, Xq, W, A, j0=0, j1=None, method="auto"):
        Xq = X if Xq is None else Xq
        Q = np.zeros(W.shape)
        j1 = W.shape[1] if j1 is None else j1
        Q[:, j0:j1] = c_oracle.quantize_layer(np.ascontiguousarray(W[:, j0:j1]), X, Xq, A)
        return Q

    def conv_layer_nhwc(self, act, actq, W, A, strides=(1, 1), padding="SAME", rate=(1, 1), c0=0, n_channels=None):
        actq = act if actq is None else actq
        kh, kw = W.shape[:2]
        rate = tuple(rate) if rate else (1, 1)

        def patches(c):
            return (O.channel_patches(act, c, (kh, kw), tuple(strides), padding, rate),
                    O.channel_patches(actq, c, (kh, kw), tuple(strides), padding, rate))
        return c_oracle.quantize_conv_layer(W, patches, A)


def _with_oracle(cls, *args, **kw):
    q = cls(*args, **kw)
    q.__class__ = type("Oracle" + cls.__name__, (cls,), {"engine": property(lambda self: OracleEngine())})
    return q


def _compare(qg, qo, x_eval, layer_kinds):
    n_checked = 0
    for idx, layer in enumerate(qg.trained_net.layers):
        if layer.__class__.__name__ not in layer_kinds:
            continue
        Wg = qg.quantized_net.layers[idx].get_weights()[0]
        Wo = qo.quantized_net.layers[idx].get_weights()[0]
        agree = float(np.mean(Wg == Wo))
        assert agree >= 0.9999, (idx, layer.__class__.__name__, agree)
        assert not np.array_equal(Wg, layer.get_weights()[0])  # the layer really was quantized
        n_checked += 1
    assert n_checked > 0
    pg, po = qg.quantized_net.predict(x_eval), qo.quantized_net.predict(x_eval)
    assert np.array_equal(pg.argmax(-1), po.argmax(-1))      # identical accuracy on any labelling of the eval set
    assert np.allclose(pg, po, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("bits,c", [(np.log2(3), 2), (4, 4)])
def test_mlp_full_network_matches_the_oracle_walk(bits, c):
    """BASELINE config 1 shape family (train_mnist_mlp.py: Flatten, Dense, BN, Dense, BN, Dense), reduced widths;
    un-normalised integer pixels with dead border features, X == Xq at the first layer."""
    rng = np.random.default_rng(11)
    net = hostnet.mnist_mlp(seed=3, widths=(96, 48), n_in=784, n_out=10)
    x = (rng.integers(0, 256, (640, 28, 28)) * (rng.random((640, 28, 28)) < 0.35)).astype(np.float32)
    x[:, :2, :] = 0
    y = rng.integers(0, 10, 640)
    seq = hostnet.ArraySequence(x, y, 160)
    qg = QuantizedNeuralNetwork(net, 160, seq, bits=bits, alphabet_scalar=c)
    qg.quantize_network()
    qo = _with_oracle(QuantizedNeuralNetwork, net, 160, seq, bits=bits, alphabet_scalar=c)
    qo.quantize_network()
    _compare(qg, qo, x[:256], {"Dense"})


@pytest.mark.parametrize("conv_path", ["nhwc", "patches"])
def test_cnn_full_network_matches_the_oracle_walk(conv_path):
    """BASELINE config 2 shape family (train_cifar10_cnn.py: 6 x Conv2D 3x3 'same' + BN / pool / dropout, 2 x Dense),
    reduced size; 4-bit alphabet; both override points of the conv path (activations vs host patch matrices)."""
    rng = np.random.default_rng(12)
    net = hostnet.cifar10_cnn(seed=5, size=16, widths=(4, 6, 8), dense=24, n_out=10)
    x = rng.random((96, 16, 16, 3)).astype(np.float32)
    y = rng.integers(0, 10, 96)
    seq = hostnet.ArraySequence(x, y, 32)
    qg = QuantizedCNN(net, 32, seq, bits=4, alphabet_scalar=4, conv_path=conv_path)
    qg.quantize_network()
    qo = _with_oracle(QuantizedCNN, net, 32, seq, bits=4, alphabet_scalar=4, conv_path="nhwc")
    qo.quantize_network()
    _compare(qg, qo, x[:64], {"Dense", "Conv2D"})


def test_cnn_with_5x5_and_7x7_kernels_through_the_default_path():
    """Kernel sizes without a dedicated kernel (the 7 x 7 / stride 2 stem of ResNet50, 5 x 5 layers) go through the default
    conv_path="nhwc" like any other: the reference handles every kernel size (quantized_network.py:686-727)."""
    rng = np.random.default_rng(14)
    L = hostnet
    net = L.Sequential([L.Conv2D(6, 7, strides=2, padding="same", activation="relu"), L.BatchNormalization(),
                        L.Conv2D(8, 5, padding="valid", activation="relu"), L.MaxPooling2D(2), L.Flatten(),
                        L.Dense(10, activation="softmax")], input_shape=(24, 24, 3), seed=4)
    x = rng.random((64, 24, 24, 3)).astype(np.float32)
    seq = hostnet.ArraySequence(x, rng.integers(0, 10, 64), 16)
    qg = QuantizedCNN(net, 16, seq, bits=3, alphabet_scalar=3)
    qg.quantize_network()
    qo = _with_oracle(QuantizedCNN, net, 16, seq, bits=3, alphabet_scalar=3)
    qo.quantize_network()
    _compare(qg, qo, x[:32], {"Dense", "Conv2D"})


@pytest.mark.parametrize("conv_path", ["nhwc", "patches"])
def test_cnn_with_non_square_strided_dilated_and_depthwise_layers(conv_path):
    """Kernels 1x3, 3x1, 2x3 and 1x2 (kk = 3, 6, 2: the patch-path kernels of those sizes), strides (2, 1) and (1, 2), dilation on
    one axis and on both, a VALID layer, and a DepthwiseConv2D with depth_multiplier 2 (its (kh, kw, C, 2) kernel is walked like a
    Conv2D kernel with two filters per channel), through both conv paths."""
    rng = np.random.default_rng(15)
    L = hostnet
    net = L.Sequential([L.Conv2D(6, (1, 3), padding="same", activation="relu"),
                        L.Conv2D(6, (3, 1), strides=(2, 1), padding="same", activation="relu"),
                        L.DepthwiseConv2D(3, padding="same", depth_multiplier=2, dilation_rate=2, activation="relu"),
                        L.Conv2D(8, (2, 3), strides=(1, 2), padding="valid", activation="relu"),
                        L.Conv2D(4, (1, 2), dilation_rate=(1, 2), padding="same", activation="relu"),
                        L.Flatten(), L.Dense(10, activation="softmax")], input_shape=(16, 16, 3), seed=4)
    x = rng.random((64, 16, 16, 3)).astype(np.float32)
    seq = hostnet.ArraySequence(x, rng.integers(0, 10, 64), 16)
    qg = QuantizedCNN(net, 16, seq, bits=3, alphabet_scalar=3, conv_path=conv_path)
    qg.quantize_network()
    qo = _with_oracle(QuantizedCNN, net, 16, seq, bits=3, alphabet_scalar=3)
    qo.quantize_network()
    _compare(qg, qo, x[:32], {"Dense", "Conv2D", "DepthwiseConv2D"})


def test_vgg_like_full_network_matches_the_oracle_walk():
    """BASELINE config 3 shape family (Keras VGG16, quantize_pretrained_imagenet.py:43-50): InputLayer, 13 conv 3x3
    'same', 5 pools, fc1 / fc2 / predictions -- a thin copy (channels / 16, 32 x 32 inputs), ternary alphabet."""
    rng = np.random.default_rng(13)
    net = hostnet.vgg16_like(seed=7, size=32, scale=16, n_out=10, fc=48)
    x = rng.random((48, 32, 32, 3)).astype(np.float32)
    seq = hostnet.ArraySequence(x, rng.integers(0, 10, 48), 16)
    qg = QuantizedCNN(net, 16, seq, bits=np.log2(3), alphabet_scalar=3)
    qg.quantize_network()
    qo = _with_oracle(QuantizedCNN, net, 16, seq, bits=np.log2(3), alphabet_scalar=3)
    qo.quantize_network()
    _compare(qg, qo, x[:32], {"Dense", "Conv2D"})


def test_grid_runner_matches_point_by_point_runs():
    """BASELINE config 5 (quantize_pretrained_cnn.py:32-48): the (bits x alphabet_scalar) grid walked in lock-step -- analog
    inputs collected once per layer, the first layer's grid points in ONE multi-alphabet call -- gives every grid point the
    weights of its own QuantizedCNN run; MSQ baselines, the CSV schema and the level-index packing of the drivers."""
    from quantized_neural_networks_b200 import QuantizedCNNGrid, get_engine, pack_levels, unpack_levels
    rng = np.random.default_rng(21)
    net = hostnet.cifar10_cnn(seed=9, size=16, widths=(4, 6, 8), dense=24, n_out=5)
    x = rng.random((96, 16, 16, 3)).astype(np.float32)
    y = rng.integers(0, 5, 96)
    seq = hostnet.ArraySequence(x, y, 32)
    quiet = type("L", (), {"info": staticmethod(lambda m: None)})()
    bits_list, scalars = [np.log2(3), 2, 4], [2, 5]
    grid = QuantizedCNNGrid(net, 32, seq, bits_list, scalars, logger=quiet).quantize_network()
    assert grid.grid == [(b, c) for b in bits_list for c in scalars]
    first = grid.calls[0]
    assert first == (first[0], len(grid.grid))               # X == Xq at the first quantized layer: one batched call
    assert all(n == 1 for _, n in grid.calls[1:])             # deeper layers: one twin, one Xq, one call per grid point
    for (b, c), qnet in zip(grid.grid, grid.quantized_nets):
        single = QuantizedCNN(net, 32, seq, logger=quiet, bits=b, alphabet_scalar=c)
        single.quantize_network()
        for idx, layer in enumerate(net.layers):
            if layer.__class__.__name__ in ("Dense", "Conv2D"):
                Wg, Ws = qnet.layers[idx].get_weights()[0], single.quantized_net.layers[idx].get_weights()[0]
                assert float(np.mean(Wg == Ws)) >= 0.9999, (b, c, idx)
                assert not np.array_equal(Wg, layer.get_weights()[0])
        assert np.array_equal(qnet.predict(x[:64]).argmax(-1), single.quantized_net.predict(x[:64]).argmax(-1))
    # MSQ baselines: plain rounding to the same per-layer alphabets (quantize_pretrained_cnn.py:97-117)
    msq = grid.msq_networks()
    for (b, c), mnet, p in zip(grid.grid, msq, grid.points):
        for idx, layer in enumerate(net.layers):
            if layer.__class__.__name__ in ("Dense", "Conv2D"):
                W = layer.get_weights()[0]
                A = O.layer_alphabet(W, c, O.unit_alphabet(b))
                ref = np.array([O.bit_round(w, A) for w in W.flatten()]).reshape(W.shape)   # the driver's own loop (:104-106)
                assert np.array_equal(np.asarray(mnet.layers[idx].get_weights()[0], dtype=np.float64), ref.astype(np.float32).astype(np.float64))
    rows = grid.metrics(x, y)
    assert len(rows) == len(grid.grid)
    assert list(rows[0]) == ["data_set", "serialized_model", "q_train_size", "ignore_layers", "bits", "alphabet_scalar",
                             "analog_test_acc", "sd_test_acc", "msq_test_acc", "quantization_time"]
    assert all(0.0 <= r["sd_test_acc"] <= 1.0 and r["q_train_size"] == 96 for r in rows)
    # int8 level indices + alphabet: the storage format of a quantized kernel
    p = grid.points[-1]
    idx_last = [i for i, l in enumerate(net.layers) if l.__class__.__name__ == "Dense"][0]
    W = net.layers[idx_last].get_weights()[0]
    Q = get_engine(0).dense_layer(x[:64].reshape(64, -1)[:, :W.shape[0]].T.copy(), None, W, np.asarray(p._layer_alphabet(W), dtype=np.float64))
    lev, A = pack_levels(Q, p._layer_alphabet(W))
    assert lev.dtype == np.int8 and np.array_equal(unpack_levels(lev, A), Q)
