"""CPU: per-channel alphabets (`alphabet_scope="channel"`) in the mirror classes, on the C oracle.

With the per-channel scope every output channel u is quantized against `rad_u * linspace(-1, 1, K)`,
`rad_u = alphabet_scalar * median(|w_u|)` -- the float32 expression of `_layer_alphabet` taken per output channel.  The GPU
tests (test_gpu_channel_alphabets.py) hold the CUDA path to the same oracle.
"""
import os
import socket

import numpy as np
import pytest

from oracle import c_oracle, channel_oracle as CO, gpfq_oracle as O
from quantized_neural_networks_b200 import QuantizedCNN, QuantizedNeuralNetwork, hostnet

QUIET = type("L", (), {"info": staticmethod(lambda m: None)})()


def with_channel_oracle(cls, *args, **kw):
    q = cls(*args, **kw)
    q.__class__ = type("ChannelOracle" + cls.__name__, (cls,), {"engine": property(lambda self: CO.ChannelOracleEngine())})
    return q


def channel_cnn(seed=6):
    """A plain 3 x 3 conv, a grouped 3 x 3 (Cg = 2), a depthwise 3 x 3 (multiplier 2) and a Dense head."""
    L = hostnet
    return L.Sequential([L.Conv2D(8, 3, padding="same", activation="relu"),
                         L.Conv2D(8, 3, padding="same", groups=4, activation="relu"),
                         L.DepthwiseConv2D(3, padding="same", depth_multiplier=2, activation="relu"),
                         L.Flatten(), L.Dense(10, activation="softmax")], input_shape=(8, 8, 3), seed=seed)


def mlp(seed=2):
    L = hostnet
    return L.Sequential([L.Dense(24, activation="relu"), L.Dense(10, activation="softmax")], input_shape=(20,), seed=seed)


def _mlp_data(n=64):
    rng = np.random.default_rng(3)
    x = rng.random((n, 20)).astype(np.float32)
    return hostnet.ArraySequence(x, rng.integers(0, 10, n), 32)


def _cnn_data(n=16):
    rng = np.random.default_rng(8)
    x = rng.random((n, 8, 8, 3)).astype(np.float32)
    return hostnet.ArraySequence(x, rng.integers(0, 10, n), 8)


@pytest.mark.parametrize("scalar", [3, 1.5, np.float64(2.0)])
def test_channel_radii_are_the_layer_expression_per_output_channel(scalar):
    net = channel_cnn()
    q = QuantizedCNN(net, 8, _cnn_data(), logger=QUIET, bits=3, alphabet_scalar=scalar, alphabet_scope="channel")
    rng = np.random.default_rng(1)
    cases = {
        "Dense": rng.standard_normal((30, 7)).astype(np.float32),
        "Conv2D": rng.standard_normal((3, 3, 4, 6)).astype(np.float32),
        "Conv2D_grouped": rng.standard_normal((3, 3, 2, 8)).astype(np.float32),        # (kh, kw, C / groups, F)
        "DepthwiseConv2D": rng.standard_normal((3, 3, 5, 2)).astype(np.float32),
    }
    for name, W in cases.items():
        kind = name.split("_")[0]
        s = q._unit_scales(W, kind)
        if kind == "Dense":
            ref = [scalar * np.median(np.abs(W[:, j].flatten())) for j in range(W.shape[1])]
            assert s.shape == (W.shape[1],)
        elif kind == "Conv2D":
            ref = [[scalar * np.median(np.abs(W[..., f].flatten())) for f in range(W.shape[3])]] * W.shape[2]
            assert s.shape == W.shape[2:]
        else:
            ref = [[scalar * np.median(np.abs(W[:, :, c, d].flatten())) for d in range(W.shape[3])] for c in range(W.shape[2])]
            assert s.shape == W.shape[2:]
        ref = np.asarray(ref)
        assert np.array_equal(s, ref.astype(np.float64)), name
        # the levels of a unit are those of the layer expression applied to the unit's own weights
        assert np.array_equal(CO.unit_levels(q.alphabet, s[0] if kind == "Dense" else s[0, 1]),
                              (ref.reshape(-1)[0 if kind == "Dense" else 1] * q.alphabet))


def test_layer_scope_is_the_default_and_reproduces_the_per_layer_run():
    net, seq = mlp(), _mlp_data()
    a = with_channel_oracle(QuantizedNeuralNetwork, net, 32, seq, logger=QUIET, bits=2, alphabet_scalar=3)
    b = with_channel_oracle(QuantizedNeuralNetwork, net, 32, seq, logger=QUIET, bits=2, alphabet_scalar=3, alphabet_scope="layer")
    assert a.alphabet_scope == "layer"
    a.quantize_network()
    b.quantize_network()
    for la, lb in zip(a.quantized_net.layers, b.quantized_net.layers):
        for wa, wb in zip(la.get_weights(), lb.get_weights()):
            assert np.array_equal(wa, wb)
    # layer scope: every Dense kernel uses the single layer alphabet
    W = net.layers[0].get_weights()[0]
    assert np.all(np.isin(a.quantized_net.layers[0].get_weights()[0], np.append(a._layer_alphabet(W), 0.0).astype(np.float32)))


@pytest.mark.parametrize("scope", ["Channel", "per-channel", "", None])
def test_bad_scope_raises(scope):
    with pytest.raises(ValueError):
        QuantizedNeuralNetwork(mlp(), 32, _mlp_data(), logger=QUIET, alphabet_scope=scope)
    with pytest.raises(ValueError):
        QuantizedCNN(channel_cnn(), 8, _cnn_data(), logger=QUIET, alphabet_scope=scope)


def test_channel_scope_uses_each_channels_own_levels():
    """Every quantized weight of a per-channel run is one of its own channel's levels (or the literal 0 of a dead
    direction), and both conv paths give the same kernels."""
    net, seq = channel_cnn(), _cnn_data()
    qs = {}
    for path in ("nhwc", "patches"):
        q = with_channel_oracle(QuantizedCNN, net, 8, seq, logger=QUIET, bits=3, alphabet_scalar=2, conv_path=path,
                                alphabet_scope="channel")
        q.quantize_network()
        qs[path] = q
    q = qs["nhwc"]
    for idx, layer in enumerate(net.layers):
        kind = layer.__class__.__name__
        if kind not in ("Dense", "Conv2D", "DepthwiseConv2D"):
            continue
        Qa = qs["nhwc"].quantized_net.layers[idx].get_weights()[0]
        assert np.array_equal(Qa, qs["patches"].quantized_net.layers[idx].get_weights()[0]), idx
        W = layer.get_weights()[0]
        s = q._unit_scales(W, kind)
        if kind == "Dense":
            for j in range(W.shape[1]):
                assert np.all(np.isin(Qa[:, j], np.append(CO.unit_levels(q.alphabet, s[j]), 0.0).astype(np.float32))), (idx, j)
        else:
            for c in range(W.shape[2]):
                for f in range(W.shape[3]):
                    lv = np.append(CO.unit_levels(q.alphabet, s[c, f]), 0.0).astype(np.float32)
                    assert np.all(np.isin(Qa[:, :, c, f], lv)), (idx, c, f)


def test_channel_scope_conv_layer_equals_the_oracle_walk():
    """The grouped layer of a per-channel run against the per-channel oracle walk on the inputs the mirror collected."""
    net, seq = channel_cnn(), _cnn_data()
    q = with_channel_oracle(QuantizedCNN, net, 8, seq, logger=QUIET, bits=3, alphabet_scalar=2, alphabet_scope="channel")
    q.quantize_network()
    data = q._get_layer_data_generator(1)
    W = net.layers[1].get_weights()[0]
    ref = CO.conv_layer(W, 4, lambda c: (O.channel_patches(data.wX, c, (3, 3), padding="SAME"),
                                          O.channel_patches(data.qX, c, (3, 3), padding="SAME")),
                        q.alphabet, q._unit_scales(W, "Conv2D"))
    assert np.array_equal(q.quantized_net.layers[1].get_weights()[0], ref.astype(np.float32))


def test_per_channel_alphabets_shrink_the_residual_of_a_layer_with_spread_scales():
    """Columns whose scales span 0.01 .. 100: one radius from the median of all columns rounds the small columns to zero and
    clips the large ones; per-channel radii keep each column's own resolution.  ||X W - X Q|| / ||X W|| over the layer (the
    first-layer form, X~ = X): 0.28 per channel against 0.97 per layer on this fixed data."""
    rng = np.random.default_rng(12)
    N0, N1, m = 64, 16, 400
    X = np.maximum(rng.standard_normal((N0, m)), 0).astype(np.float32)
    W = (rng.standard_normal((N0, N1)) * np.logspace(-2, 2, N1)).astype(np.float32)
    A = O.unit_alphabet(3)
    Q_layer = c_oracle.quantize_layer(W, X, X, 2 * np.median(np.abs(W.flatten())) * A)
    Q_chan = CO.dense_layer(W, X, X, A, (2 * np.median(np.abs(W), axis=0)).astype(np.float64))
    Xd = X.T.astype(np.float64)
    rel = lambda Q: np.linalg.norm(Xd @ W - Xd @ Q) / np.linalg.norm(Xd @ W)
    assert rel(Q_chan) < 0.5 * rel(Q_layer), (rel(Q_chan), rel(Q_layer))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _channel_shard_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        net, seq = channel_cnn(), _cnn_data()
        ok = True
        for path in ("nhwc", "patches"):
            kw = dict(logger=QUIET, bits=2, alphabet_scalar=3, conv_path=path, alphabet_scope="channel")
            one = with_channel_oracle(QuantizedCNN, net, 8, seq, **kw)
            one.quantize_network()
            shr = with_channel_oracle(QuantizedCNN, net, 8, seq, shard=(rank, world), **kw)
            shr.quantize_network()
            for idx in (0, 1, 2, 4):
                ok = ok and np.array_equal(one.quantized_net.layers[idx].get_weights()[0],
                                           shr.quantized_net.layers[idx].get_weights()[0])
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_channel_shards_of_a_per_channel_run_are_gathered(world):
    """Channel, group and neuron shards of a per-channel run, all-gathered under gloo, equal the one-rank run."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_channel_shard_worker, args=(r, world, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    assert dict(ret) == {r: True for r in range(world)}


def test_pack_unpack_round_trip_with_per_channel_scales():
    """Level indices of a per-channel kernel refer to each unit's own levels fl64(s_u * A[k]); unpacking with the same scales gives
    the kernel back bit for bit, the literal 0 of a dead direction included.  Without scales the call is the per-layer one."""
    from quantized_neural_networks_b200 import pack_levels, unpack_levels
    rng = np.random.default_rng(7)
    A = O.unit_alphabet(3)
    for shape in ((40, 6), (3, 3, 4, 5)):
        units = shape[-1:] if len(shape) == 2 else shape[-2:]
        s = (10.0 ** rng.uniform(-2, 2, units)).astype(np.float32).astype(np.float64)
        s.reshape(-1)[1] = 0.0                                    # a zero scale: all levels are 0
        k = rng.integers(0, len(A), shape)
        Q = np.take_along_axis(np.broadcast_to(s[..., None] * A, shape + (len(A),)), k[..., None], -1)[..., 0]
        Q.reshape(-1)[0] = 0.0                                    # a dead direction
        idx, base = pack_levels(Q, A, scales=s)
        assert idx.dtype == np.int8 and np.array_equal(base, A)
        assert np.array_equal(unpack_levels(idx, A, scales=s), Q)
        with pytest.raises(ValueError):
            pack_levels(Q, A, scales=s[..., :-1])
    Ql = rng.choice(2.5 * A, (8, 3))
    assert np.array_equal(unpack_levels(*pack_levels(Ql, 2.5 * A)), Ql)
