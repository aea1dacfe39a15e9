"""CPU: grouped Conv2D (`groups` > 1) in the host layers and the mirror classes.

A grouped kernel is (kh, kw, C / groups, F): filter f of group g = f // Fg (Fg = F / groups) reads only the input channels
g Cg .. (g + 1) Cg - 1 (Cg = C / groups).  The GPFQ problem of such a layer is the per-(input channel, filter) walk with input
channel c paired only with the Fg filters of its own group.  `grouped_oracle_conv` states that walk with the literal C oracle;
the GPU tests (test_gpu_conv_groups.py) hold the CUDA path to it.
"""
import os
import socket

import numpy as np
import pytest

from oracle import c_oracle, gpfq_oracle as O
from quantized_neural_networks_b200 import QuantizedCNN, hostnet
from quantized_neural_networks_b200.replicate import shard_range

QUIET = type("L", (), {"info": staticmethod(lambda m: None)})()


def grouped_oracle_conv(W, groups, patches, A, c0=0, n_channels=None):
    """Literal walk of input channels c0 .. c0+n_channels-1 of a grouped (kh, kw, C / groups, F) kernel: channel c against the
    Fg filters of its group only.  `patches(c) -> (Xp, Xqp)`, each (kh*kw, n).  Other entries stay 0."""
    kh, kw, Cg, F = W.shape
    Fg = F // groups
    n_channels = Cg * groups - c0 if n_channels is None else n_channels
    Q = np.zeros(W.shape)
    for c in range(c0, c0 + n_channels):
        ci, f0 = c % Cg, (c // Cg) * Fg
        Xp, Xqp = patches(c)
        Wc = np.ascontiguousarray(W[:, :, ci, f0:f0 + Fg].reshape(kh * kw, Fg))
        Q[:, :, ci, f0:f0 + Fg] = c_oracle.quantize_layer(Wc, Xp, Xqp, A).reshape(kh, kw, Fg)
    return Q


class GroupedOracleEngine:
    """The engine's call surface (with `groups`) routed through the C oracle."""
    last_stats = {}

    def dense_layer(self, X, Xq, W, A, j0=0, j1=None, method="auto"):
        Q = np.zeros(W.shape)
        j1 = W.shape[1] if j1 is None else j1
        Q[:, j0:j1] = c_oracle.quantize_layer(np.ascontiguousarray(W[:, j0:j1]), X, X if Xq is None else Xq, A)
        return Q

    def conv_channels(self, Xp, Xqp, W, A, c0=0, n_channels=None):
        kh, kw, C, F = W.shape
        Q = np.zeros(W.shape)
        for i in range(C):
            Wc = np.ascontiguousarray(W[:, :, i, :].reshape(kh * kw, F))
            Q[:, :, i, :] = c_oracle.quantize_layer(Wc, Xp[i], Xp[i] if Xqp is None else Xqp[i], A).reshape(kh, kw, F)
        return Q

    def conv_layer_nhwc(self, act, actq, W, A, strides=(1, 1), padding="SAME", rate=(1, 1), c0=0, n_channels=None, groups=1):
        actq = act if actq is None else actq
        ks = tuple(W.shape[:2])
        rate = tuple(rate) if rate else (1, 1)

        def patches(c):
            return (O.channel_patches(act, c, ks, tuple(strides), padding, rate),
                    O.channel_patches(actq, c, ks, tuple(strides), padding, rate))
        return grouped_oracle_conv(W, groups, patches, A, c0, n_channels)


def with_grouped_oracle(cls, *args, **kw):
    q = cls(*args, **kw)
    q.__class__ = type("GroupedOracle" + cls.__name__, (cls,), {"engine": property(lambda self: GroupedOracleEngine())})
    return q


def grouped_cnn(seed=4):
    """ResNeXt / RegNet-style 3 x 3 (Cg = 4), ShuffleNet-style 1 x 1 (groups 8), ConvNeXt-style 7 x 7 with groups = C, and a
    strided 5 x 5 with Cg = 8."""
    L = hostnet
    return L.Sequential([L.Conv2D(16, 3, padding="same", activation="relu"),
                         L.Conv2D(16, 3, padding="same", groups=4, activation="relu"),
                         L.Conv2D(24, 1, groups=8, activation="relu"),
                         L.Conv2D(24, 7, padding="same", groups=24, activation="relu"),
                         L.Conv2D(12, 5, strides=2, padding="valid", groups=3, activation="relu"),
                         L.Flatten(), L.Dense(10, activation="softmax")], input_shape=(14, 14, 3), seed=seed)


def _torch_conv(x, W, strides, padding, rate, groups):
    """torch.nn.functional.conv2d on NHWC input with an explicit TensorFlow-style SAME padding."""
    import torch
    import torch.nn.functional as tF
    kh, kw = W.shape[:2]
    xt = torch.from_numpy(np.ascontiguousarray(x.transpose(0, 3, 1, 2))).double()
    if padding == "same":
        H, Wd = x.shape[1:3]
        _, pt, pb = hostnet._same_pad(H, (kh - 1) * rate[0] + 1, strides[0])
        _, pl, pr = hostnet._same_pad(Wd, (kw - 1) * rate[1] + 1, strides[1])
        xt = tF.pad(xt, (pl, pr, pt, pb))
    wt = torch.from_numpy(np.ascontiguousarray(W.transpose(3, 2, 0, 1))).double()   # (F, C / groups, kh, kw)
    y = tF.conv2d(xt, wt, stride=strides, dilation=rate, groups=groups)
    return y.numpy().transpose(0, 2, 3, 1)


@pytest.mark.parametrize("filters,ks,strides,padding,rate,groups,c_in", [
    (16, 3, (1, 1), "same", (1, 1), 4, 16),
    (9, 1, (1, 1), "valid", (1, 1), 3, 6),
    (12, 7, (1, 1), "same", (1, 1), 12, 12),
    (10, 5, (2, 1), "same", (2, 1), 2, 6),
    (6, (3, 2), (1, 2), "valid", (1, 1), 6, 6),
])
def test_grouped_forward_matches_torch(filters, ks, strides, padding, rate, groups, c_in):
    rng = np.random.default_rng(filters * 7 + groups)
    layer = hostnet.Conv2D(filters, ks, strides=strides, padding=padding, dilation_rate=rate, groups=groups, use_bias=False)
    net = hostnet.Sequential([layer], input_shape=(11, 12, c_in), seed=2)
    W = layer.get_weights()[0]
    assert W.shape == (*layer.kernel_size, c_in // groups, filters)
    x = rng.standard_normal((3, 11, 12, c_in)).astype(np.float32)
    y = net.predict(x)
    ref = _torch_conv(x.astype(np.float64), W.astype(np.float64), strides, padding, rate, groups)
    assert y.shape == ref.shape
    assert np.allclose(y, ref, rtol=1e-5, atol=1e-5)


def test_groups_equal_to_channels_is_a_depthwise_layer():
    """Conv2D(groups=C, filters=C*M) computes DepthwiseConv2D(depth_multiplier=M) with the kernel (kh, kw, C, M) stored as
    (kh, kw, 1, C*M)."""
    rng = np.random.default_rng(5)
    C, M = 5, 2
    dw = hostnet.DepthwiseConv2D(3, padding="same", depth_multiplier=M, use_bias=False)
    gc = hostnet.Conv2D(C * M, 3, padding="same", groups=C, use_bias=False)
    ndw = hostnet.Sequential([dw], input_shape=(9, 9, C), seed=1)
    ngc = hostnet.Sequential([gc], input_shape=(9, 9, C), seed=1)
    Wd = dw.get_weights()[0]
    ngc.set_weights([Wd.reshape(3, 3, 1, C * M)])
    x = rng.standard_normal((2, 9, 9, C)).astype(np.float32)
    assert np.allclose(ngc.predict(x), ndw.predict(x), rtol=1e-6, atol=1e-6)


def test_bad_groups_are_rejected_by_the_layer():
    with pytest.raises(ValueError):
        hostnet.Sequential([hostnet.Conv2D(8, 3, groups=3)], input_shape=(6, 6, 6))   # 8 filters
    with pytest.raises(ValueError):
        hostnet.Sequential([hostnet.Conv2D(6, 3, groups=3)], input_shape=(6, 6, 4))   # 4 input channels


def test_clone_model_keeps_groups():
    net = grouped_cnn()
    clone = hostnet.clone_model(net)
    for a, b in zip(net.layers, clone.layers):
        assert getattr(a, "groups", None) == getattr(b, "groups", None)
        assert [w.shape for w in a.get_weights()] == [w.shape for w in b.get_weights()]
    assert clone.layers[3].groups == 24 and clone.layers[3].get_weights()[0].shape == (7, 7, 1, 24)


def _cnn_data(n=32):
    rng = np.random.default_rng(8)
    x = rng.random((n, 14, 14, 3)).astype(np.float32)
    return x, hostnet.ArraySequence(x, rng.integers(0, 10, n), 16)


def test_mirror_quantizes_grouped_layers_the_same_through_both_conv_paths():
    """The nhwc path hands the whole grouped layer to the engine (`groups=`); the patches path walks channel c with the kernel
    slice W[:, :, c % Cg, g Fg:(g + 1) Fg].  On the oracle engine both give the same kernels, and each grouped layer equals the
    grouped oracle walk on its own inputs."""
    net = grouped_cnn()
    x, seq = _cnn_data()
    qs = {}
    for path in ("nhwc", "patches"):
        q = with_grouped_oracle(QuantizedCNN, net, 16, seq, logger=QUIET, bits=3, alphabet_scalar=3, conv_path=path)
        q.quantize_network()
        qs[path] = q
    n_grouped = 0
    for idx, layer in enumerate(net.layers):
        if layer.__class__.__name__ in ("Conv2D", "Dense"):
            a = qs["nhwc"].quantized_net.layers[idx].get_weights()[0]
            b = qs["patches"].quantized_net.layers[idx].get_weights()[0]
            assert np.array_equal(a, b), idx
            assert not np.array_equal(a, layer.get_weights()[0]), idx
            n_grouped += getattr(layer, "groups", 1) > 1
    assert n_grouped == 4
    # the 1 x 1 layer (groups 8) against the oracle walk on the inputs the mirror collected
    q = qs["nhwc"]
    data = q._get_layer_data_generator(2)
    W = net.layers[2].get_weights()[0]
    A = q._layer_alphabet(W)
    ref = grouped_oracle_conv(W, 8, lambda c: (O.channel_patches(data.wX, c, (1, 1)), O.channel_patches(data.qX, c, (1, 1))), A)
    assert np.array_equal(q.quantized_net.layers[2].get_weights()[0], ref.astype(np.float32))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _group_shard_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        net = hostnet.Sequential([hostnet.Conv2D(6, 3, padding="same", activation="relu"),
                                  hostnet.Conv2D(12, 3, padding="same", groups=3, activation="relu"),
                                  hostnet.Conv2D(4, 1, groups=2, activation="relu"),
                                  hostnet.Flatten(), hostnet.Dense(5, activation="softmax")], input_shape=(8, 8, 3), seed=3)
        rng = np.random.default_rng(2)
        seq = hostnet.ArraySequence(rng.random((16, 8, 8, 3)).astype(np.float32), np.zeros(16), 8)
        ok = True
        for path in ("nhwc", "patches"):
            one = with_grouped_oracle(QuantizedCNN, net, 8, seq, logger=QUIET, bits=2, alphabet_scalar=3, conv_path=path)
            one.quantize_network()
            shr = with_grouped_oracle(QuantizedCNN, net, 8, seq, logger=QUIET, bits=2, alphabet_scalar=3, conv_path=path,
                                      shard=(rank, world))
            shr.quantize_network()
            for idx in (1, 2):
                ok = ok and np.array_equal(one.quantized_net.layers[idx].get_weights()[0],
                                           shr.quantized_net.layers[idx].get_weights()[0])
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_group_shards_are_gathered_along_the_filter_axis(world):
    """Ranks take whole groups (3 groups over 2 or 3 ranks; 2 groups over 3 ranks leaves one rank without a group) and the
    all-gather puts each rank's filters back: the sharded run equals the one-rank run, through both conv paths."""
    import torch.multiprocessing as mp
    assert [shard_range(2, r, 3) for r in range(3)] == [(0, 1), (1, 2), (2, 2)]
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_group_shard_worker, args=(r, world, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    assert dict(ret) == {r: True for r in range(world)}
