"""GPU: per-channel alphabets (the `*_scaled` entry points): unit u walks with the levels fl64(s_u * A[k]).

The checker is the literal C oracle run one unit at a time with that unit's own levels (oracle/channel_oracle.py), entry for
entry; every other way into the same layer (host arrays, device tensors, channel shards, the Gram-only pair, batched
alphabets) must give the same bits.
"""
from ctypes import POINTER, byref, c_double, c_int32, c_void_p

import numpy as np
import pytest

from conftest import glorot, golden, hidden_pair
from oracle import channel_oracle as CO, gpfq_oracle as O
from quantized_neural_networks_b200 import GpfqError, QuantizedCNN, QuantizedNeuralNetwork, _lib, hostnet
from quantized_neural_networks_b200.grid import QuantizedCNNGrid
from test_host_channel_alphabets import QUIET, channel_cnn, mlp, with_channel_oracle

pytestmark = pytest.mark.gpu


def _scales(rng, shape, zero_at=None):
    """Seeded scales spanning 0.01 .. 100 (float32 values, as radii are), one of them 0."""
    s = (10.0 ** rng.uniform(-2, 2, shape)).astype(np.float32).astype(np.float64)
    if zero_at is not None:
        s[zero_at] = 0.0
    return s


@pytest.fixture
def options(engine):
    """Set engine options for one test and restore the defaults after it."""
    touched = []

    def set_(**kw):
        for k, v in kw.items():
            engine.set_option(k, v)
            touched.append(k)
    yield set_
    for k in touched:
        engine.set_option(k, 0)


# name: (N0, N1, m, bits, method, options, dead directions, stats.reserved: bit 0 int8 residual form, bit 1 tensor-core walk)
DENSE = {
    "stream_ternary": (96, 45, 300, np.log2(3), "stream", {}, 3, 0),
    "stream_fast_4bit": (96, 45, 300, 4, "stream_fast", {}, 3, 0),
    "stream_long_m": (40, 9, 9000, 2, "stream", {}, 2, 0),                     # residual in shared memory
    "tile_pipe_ternary": (300, 200, 500, np.log2(3), "gram", {"sweep_walk": 2}, 4, 0),
    "tile_pipe_2bit": (300, 200, 500, 2, "gram", {"sweep_walk": 2}, 4, 0),
    "tile_pipe_6bit": (300, 131, 500, 6, "gram", {"sweep_walk": 2}, 4, 0),
    "tile_many_neurons": (160, 2100, 200, 3, "gram", {"sweep_walk": 2}, 2, 0),   # 32-neuron tiles
    "tc_ternary": (300, 131, 500, np.log2(3), "gram", {"sweep_walk": 1, "sweep_outer": 1}, 4, 2),
    "tc_2bit": (300, 131, 500, 2, "gram", {"sweep_walk": 1, "sweep_outer": 1}, 4, 2),
    "tc_4bit": (300, 131, 500, 4, "gram", {"sweep_walk": 1, "sweep_outer": 1}, 4, 2),
    "tc_6bit": (300, 131, 500, 6, "gram", {"sweep_walk": 1, "sweep_outer": 1}, 4, 2),
    "residual_i8_ternary": (1100, 70, 160, np.log2(3), "gram", {"sweep_outer": 2, "sweep_i8": 1}, 5, 3),
    "residual_i8_4bit": (1100, 70, 160, 4, "gram", {"sweep_outer": 2, "sweep_i8": 1}, 5, 3),
    "residual_fp64_2bit": (1100, 70, 160, 2, "gram", {"sweep_outer": 2, "sweep_i8": 2}, 5, 0),
    "residual_two_chains": (1100, 2100, 160, np.log2(3), "gram", {"sweep_outer": 2}, 5, 3),
}


@pytest.mark.parametrize("name", list(DENSE))
def test_dense_scaled_matches_the_oracle_unit_by_unit(engine, options, name):
    N0, N1, m, bits, method, opts, dead, reserved = DENSE[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    X, Xq = hidden_pair(rng, N0, m)
    X[:dead] = 0.0
    Xq[:dead] = 0.0                       # dead directions: the literal 0
    W = glorot(rng, N0, N1)
    A = O.unit_alphabet(bits)
    s = _scales(rng, N1, zero_at=1) * float(np.median(np.abs(W)))
    options(**opts)
    Q = engine.dense_layer(X, Xq, W, A, method=method, scales=s)
    st = dict(engine.last_stats)
    cols = range(N1) if N1 <= 200 else list(range(0, N1, 97)) + [N1 - 1]
    ref = CO.dense_layer(W, X, Xq, A, s, cols=cols)
    cols = list(cols)
    assert np.array_equal(Q[:, cols], ref[:, cols]), (name, st)
    assert np.all(Q[:, 1] == 0.0)          # zero scale: all-zero column
    assert st["reserved"] & 3 == reserved, (name, st)   # the fast kernel the case is named for actually ran


@pytest.mark.parametrize("name", ["dense_first_ternary", "dense_hidden_grid", "ties_and_dead"])
def test_golden_dense_vectors_with_scales(engine, options, name):
    g = golden(name)
    X = g["X"]
    Xq = g["Xq"] if "Xq" in g.files else None
    W = g["W"]
    rng = np.random.default_rng(5)
    s = _scales(rng, W.shape[1], zero_at=0) * float(np.median(np.abs(W)))
    A = O.unit_alphabet(np.log2(3))
    ref = CO.dense_layer(W, X, X if Xq is None else Xq, A, s)
    for method in ("stream", "gram"):
        assert np.array_equal(engine.dense_layer(X, Xq, W, A, method=method, scales=s), ref), method
    options(sweep_walk=1)
    for outer in (1, 2):                  # the tensor-core walk: Gram rows, carried residuals
        options(sweep_outer=outer)
        Q = engine.dense_layer(X, Xq, W, A, method="gram", scales=s)
        assert engine.last_stats["reserved"] & 2, engine.last_stats
        assert np.array_equal(Q, ref), outer


@pytest.mark.parametrize("case", ["stream", "gram_tile", "vgg_fc1_shape", "gram_rows_4096"])
def test_uniform_scales_equal_the_per_layer_call(engine, options, case):
    """Every scale equal to rad with the base alphabet linspace(-1, 1, K) is the per-layer alphabet rad * linspace: same bits."""
    rng = np.random.default_rng(len(case))
    N0, N1, m, method, opts = {"stream": (200, 60, 400, "stream", {}),
                               "gram_tile": (400, 150, 600, "gram", {"sweep_walk": 2}),
                               "vgg_fc1_shape": (4096, 256, 600, "gram", {}),
                               "gram_rows_4096": (4096, 128, 6000, "gram", {"sweep_outer": 1})}[case]
    X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    base = O.unit_alphabet(np.log2(3))
    rad = np.float32(3) * np.median(np.abs(W.flatten()))
    options(**opts)
    Q1 = engine.dense_layer(X, Xq, W, rad * base, method=method)
    st1 = dict(engine.last_stats)
    Q2 = engine.dense_layer(X, Xq, W, base, method=method, scales=np.full(N1, float(rad)))
    st2 = dict(engine.last_stats)
    assert np.array_equal(Q1, Q2), (st1, st2)
    assert st1["gram_kernel"] == st2["gram_kernel"] and st1["reserved"] == st2["reserved"], (st1, st2)
    expect = {"stream": 0, "gram_tile": 0, "vgg_fc1_shape": 3, "gram_rows_4096": 2}[case]
    assert st2["reserved"] & 3 == expect, st2     # bits 0 | 1 on the fc1 shape, bit 1 on the 4096-direction Gram-row call


def test_vgg_fc1_full_size_per_channel(engine):
    """VGG16 fc1 shape (N0 = 25088, m = 1504: the residual form), 512 neurons with their own radii; sampled neurons against
    the oracle."""
    rng = np.random.default_rng(31)
    N0, N1, m = 25088, 512, 1504
    X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1) * np.logspace(-1, 1, N1, dtype=np.float32)
    A = O.unit_alphabet(np.log2(3))
    s = (np.float32(3) * np.median(np.abs(W), axis=0)).astype(np.float64)
    Q = engine.dense_layer(X, Xq, W, A, scales=s)
    st = dict(engine.last_stats)
    assert st["gram_kernel"] == 3 and st["reserved"] & 3 == 3, st     # the residual form with its contractions on tcgen05
    cols = [0, 1, 200, 511]
    assert O.agreement(Q[:, cols], CO.dense_layer(W, X, Xq, A, s, cols=cols)[:, cols]) >= 0.9999


def test_dense_from_gram_and_shards_with_scales(engine):
    import torch
    rng = np.random.default_rng(9)
    N0, N1, m = 300, 90, 700
    X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    A = O.unit_alphabet(3)
    s = _scales(rng, N1, zero_at=7) * float(np.median(np.abs(W)))
    ref = CO.dense_layer(W, X, Xq, A, s)
    G1, G2 = engine.gram_matrices(torch.from_numpy(X).cuda(), torch.from_numpy(Xq).cuda())
    assert np.array_equal(engine.dense_layer_from_gram(G1, G2, W, A, scales=s), ref)
    Qs = np.zeros_like(ref)
    for j0, j1 in ((0, 31), (31, 64), (64, 90)):
        Qs[:, j0:j1] = engine.dense_layer(X, Xq, W, A, j0=j0, j1=j1, method="gram", scales=torch.tensor(s))[:, j0:j1]
    assert np.array_equal(Qs, ref)
    Qd = engine.dense_layer(torch.from_numpy(X).cuda(), torch.from_numpy(Xq).cuda(), torch.from_numpy(W).cuda(), A, scales=s)
    assert np.array_equal(Qd.cpu().numpy(), ref)


def test_dense_alphabet_batching_with_scales(engine):
    rng = np.random.default_rng(10)
    N0, N1, m = 300, 70, 500
    X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    As = [O.unit_alphabet(b) for b in (np.log2(3), 2, 4)]
    S = np.stack([_scales(rng, N1, zero_at=a) * float(np.median(np.abs(W))) for a in range(3)])
    for method in ("stream", "gram"):
        Qb = engine.dense_layer(X, Xq, W, As, method=method, scales=S)
        for a in range(3):
            assert np.array_equal(Qb[a], engine.dense_layer(X, Xq, W, As[a], method=method, scales=S[a])), (method, a)


# (kernel, strides, rate, padding, (n_img, H, W), C, F, groups, bits)
CONV = {
    "1x1": ((1, 1), (1, 1), (1, 1), "VALID", (4, 8, 9), 6, 9, 1, 2),
    "2x1": ((2, 1), (1, 1), (1, 1), "VALID", (4, 8, 9), 5, 7, 1, 3),
    "1x3": ((1, 3), (1, 1), (1, 1), "SAME", (4, 8, 9), 5, 7, 1, 3),
    "2x2": ((2, 2), (1, 1), (1, 1), "VALID", (4, 8, 9), 5, 7, 1, 4),
    "2x3": ((2, 3), (1, 1), (1, 1), "SAME", (4, 8, 9), 5, 7, 1, 3),
    "3x3_c32_corr": ((3, 3), (1, 1), (1, 1), "SAME", (4, 12, 12), 32, 12, 1, np.log2(3)),
    "3x3_stride2": ((3, 3), (2, 2), (1, 1), "SAME", (4, 13, 12), 6, 140, 1, 3),
    "5x5": ((5, 5), (1, 1), (1, 1), "SAME", (4, 10, 10), 4, 6, 1, 3),
    "7x7": ((7, 7), (1, 1), (1, 1), "SAME", (4, 10, 11), 4, 20, 1, 2),
    "13x11_fallback": ((13, 11), (1, 1), (1, 1), "SAME", (2, 14, 13), 3, 5, 1, 3),
    "3x3_grouped": ((3, 3), (1, 1), (1, 1), "SAME", (4, 12, 12), 8, 12, 2, 3),
    "7x7_depthwise": ((7, 7), (1, 1), (1, 1), "SAME", (4, 10, 11), 6, 12, 6, 3),
    "3x3_depthwise_32": ((3, 3), (1, 1), (1, 1), "SAME", (4, 10, 10), 32, 32, 32, np.log2(3)),
}


def _conv(name):
    ks, strides, rate, pad, (n_img, H, Wd), C, F, groups, bits = CONV[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    W = (rng.uniform(-1, 1, (*ks, C // groups, F)) * 0.4).astype(np.float32)
    s = _scales(rng, W.shape[2:], zero_at=(0, 1)) * float(np.median(np.abs(W)))
    geo = dict(strides=strides, padding=pad, rate=rate)
    patches = lambda c: (O.channel_patches(act, c, ks, **geo), O.channel_patches(actq, c, ks, **geo))
    return ks, geo, act, actq, W, O.unit_alphabet(bits), s, groups, patches


@pytest.mark.parametrize("name", list(CONV))
def test_conv_scaled_matches_the_oracle_every_entry_path(engine, name):
    import torch
    ks, geo, act, actq, W, A, s, groups, patches = _conv(name)
    gk = {"groups": groups} if groups > 1 else {}
    ref = CO.conv_layer(W, groups, patches, A, s)
    Q = engine.conv_layer_nhwc(act, actq, W, A, scales=s, **geo, **gk)
    assert np.array_equal(Q, ref), name
    assert np.all(Q[:, :, 0, 1] == 0.0)
    cuda = lambda a: torch.from_numpy(a).cuda()
    Qd = engine.conv_layer_nhwc(cuda(act), cuda(actq), cuda(W), A, scales=torch.tensor(s), **geo, **gk).cpu().numpy()
    assert np.array_equal(Qd, ref), name
    C = act.shape[3]
    c0, n_ch = (1, C - 2) if groups == 1 else (W.shape[2] // 2, W.shape[2])   # a shard that crosses a group
    Qs = engine.conv_layer_nhwc(act, actq, W, A, scales=s, c0=c0, n_channels=n_ch, **geo, **gk)
    own = CO.conv_layer(W, groups, patches, A, s, c0, n_ch)
    assert np.array_equal(Qs, own), name
    if groups == 1:
        Qc = engine.conv_channels([patches(c)[0] for c in range(C)], [patches(c)[1] for c in range(C)], W, A, scales=s)
        assert np.array_equal(Qc, ref), name
    if ks[0] * ks[1] <= 128:
        n_img = act.shape[0]
        gram = (engine.conv_gram_nhwc(act[:n_img // 2], actq[:n_img // 2], ks, **geo)
                + engine.conv_gram_nhwc(act[n_img // 2:], actq[n_img // 2:], ks, **geo))
        assert np.array_equal(engine.conv_layer_from_gram(gram, W, A, scales=s, **gk), ref), name


@pytest.mark.parametrize("name", ["3x3_c32_corr", "7x7", "3x3_grouped"])
def test_conv_uniform_scales_equal_the_per_layer_call(engine, name):
    ks, geo, act, actq, W, A, s, groups, patches = _conv(name)
    gk = {"groups": groups} if groups > 1 else {}
    rad = np.float32(2) * np.median(np.abs(W.flatten()))
    Q1 = engine.conv_layer_nhwc(act, actq, W, rad * A, **geo, **gk)
    k1 = engine.last_stats["gram_kernel"]
    Q2 = engine.conv_layer_nhwc(act, actq, W, A, scales=np.full(W.shape[2:], float(rad)), **geo, **gk)
    assert np.array_equal(Q1, Q2) and engine.last_stats["gram_kernel"] == k1


def test_conv_alphabet_batching_with_scales(engine):
    ks, geo, act, actq, W, _, s, groups, patches = _conv("5x5")
    As = [O.unit_alphabet(b) for b in (np.log2(3), 2, 4)]
    S = np.stack([s * (a + 1) for a in range(3)])
    Qb = engine.conv_layer_nhwc(act, actq, W, As, scales=S, **geo)
    for a in range(3):
        assert np.array_equal(Qb[a], engine.conv_layer_nhwc(act, actq, W, As[a], scales=S[a], **geo)), a


def test_msq_per_channel_equals_numpy(engine):
    rng = np.random.default_rng(4)
    A = O.unit_alphabet(3)
    for W in (rng.standard_normal((40, 13)).astype(np.float32), rng.standard_normal((3, 3, 4, 6)).astype(np.float32)):
        s = _scales(rng, W.shape[-1:] if W.ndim == 2 else W.shape[-2:], zero_at=0)
        assert np.array_equal(engine.msq(W, A, scales=s), CO.msq(W, A, s))


def test_bad_scales_raise_and_return_err_arg(engine):
    rng = np.random.default_rng(2)
    X, Xq = hidden_pair(rng, 20, 50)
    W = glorot(rng, 20, 6)
    A = O.unit_alphabet(2)
    for bad in (np.ones(5), np.array([1, 1, -1, 1, 1, 1.0]), np.array([1, np.nan, 1, 1, 1, 1.0]), np.full(6, np.inf)):
        with pytest.raises(ValueError):
            engine.dense_layer(X, Xq, W, A, scales=bad)
    with pytest.raises(ValueError):
        engine.conv_layer_nhwc(np.ones((1, 4, 4, 2), np.float32), None, np.ones((3, 3, 2, 3), np.float32), A, scales=np.ones((3, 2)))
    lib = _lib.lib()
    Q = np.zeros((20, 6))
    K = np.array([len(A)], np.int32)
    for bad in (np.array([1, 1, -1, 1, 1, 1.0]), np.array([1, np.nan, 1, 1, 1, 1.0])):
        st = _lib.GpfqStats()
        engine._bind_stream(False)
        rc = lib.gpfq_dense_layer_scaled(engine._ctx, c_void_p(X.ctypes.data), c_void_p(Xq.ctypes.data), 50, 20, 50,
                                         c_void_p(W.ctypes.data), 6, 6, 0, 6, A.ctypes.data_as(POINTER(c_double)),
                                         K.ctypes.data_as(POINTER(c_int32)), 1, c_void_p(Q.ctypes.data), 6, 0, byref(st),
                                         bad.ctypes.data_as(POINTER(c_double)))
        assert rc == 1
        rc = lib.gpfq_msq_scaled(engine._ctx, c_void_p(W.ctypes.data), W.size, A.ctypes.data_as(POINTER(c_double)), len(A),
                                 bad.ctypes.data_as(POINTER(c_double)), 6, c_void_p(Q.ctypes.data), 0)
        assert rc == 1
    with pytest.raises(GpfqError):
        engine._check(1)


def _predict_equal(a, b, x):
    return np.array_equal(a.predict(x), b.predict(x))


def test_networks_with_channel_scope_match_the_mirror(engine):
    rng = np.random.default_rng(3)
    xm = rng.random((64, 20)).astype(np.float32)
    seq = hostnet.ArraySequence(xm, rng.integers(0, 10, 64), 32)
    net = mlp()
    gpu = QuantizedNeuralNetwork(net, 32, seq, logger=QUIET, bits=2, alphabet_scalar=3, alphabet_scope="channel")
    ref = with_channel_oracle(QuantizedNeuralNetwork, net, 32, seq, logger=QUIET, bits=2, alphabet_scalar=3,
                              alphabet_scope="channel")
    gpu.quantize_network()
    ref.quantize_network()
    for la, lb in zip(gpu.quantized_net.layers, ref.quantized_net.layers):
        for wa, wb in zip(la.get_weights(), lb.get_weights()):
            assert np.array_equal(wa, wb)
    assert _predict_equal(gpu.quantized_net, ref.quantized_net, xm)
    cnn = channel_cnn()
    xc = np.random.default_rng(8).random((16, 8, 8, 3)).astype(np.float32)
    seqc = hostnet.ArraySequence(xc, np.zeros(16), 8)
    mirror = with_channel_oracle(QuantizedCNN, cnn, 8, seqc, logger=QUIET, bits=3, alphabet_scalar=2, alphabet_scope="channel")
    mirror.quantize_network()
    for path in ("nhwc", "patches"):
        q = QuantizedCNN(cnn, 8, seqc, logger=QUIET, bits=3, alphabet_scalar=2, conv_path=path, alphabet_scope="channel")
        q.quantize_network()
        for la, lb in zip(q.quantized_net.layers, mirror.quantized_net.layers):
            for wa, wb in zip(la.get_weights(), lb.get_weights()):
                assert np.array_equal(wa, wb), path
        assert _predict_equal(q.quantized_net, mirror.quantized_net, xc)
    grid = QuantizedCNNGrid(cnn, 8, seqc, [2, 3], [2, 3], logger=QUIET, alphabet_scope="channel").quantize_network()
    for (bits, c), p in zip(grid.grid, grid.points):
        one = with_channel_oracle(QuantizedCNN, cnn, 8, seqc, logger=QUIET, bits=bits, alphabet_scalar=c, alphabet_scope="channel")
        one.quantize_network()
        for la, lb in zip(p.quantized_net.layers, one.quantized_net.layers):
            for wa, wb in zip(la.get_weights(), lb.get_weights()):
                assert np.array_equal(wa, wb), (bits, c)
    for (bits, c), p, msq in zip(grid.grid, grid.points, grid.msq_networks()):
        W = cnn.layers[0].get_weights()[0]
        A, s = p._levels(W, "Conv2D")
        assert np.array_equal(msq.layers[0].get_weights()[0], CO.msq(W, A, s).astype(np.float32))
