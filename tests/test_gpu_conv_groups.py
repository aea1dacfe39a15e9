"""GPU: grouped Conv2D layers (`groups` > 1: ResNeXt, RegNet, ConvNeXt's Conv2D(groups=C), ShuffleNet) through the batched conv
path in one call (`gpfq_conv_layer_nhwc_grouped`, `gpfq_conv_layer_from_gram_grouped`).

The kernel is (kh, kw, C / groups, F) and input channel c is walked against the Fg = F / groups filters of its own group only.
The checker is the literal C oracle walked that way (`grouped_oracle_conv`, test_host_conv_groups.py), entry for entry; every
other way into the same layer must give the same bits.
"""
from ctypes import POINTER, c_double, c_int32, c_void_p

import numpy as np
import pytest

from oracle import gpfq_oracle as O
from quantized_neural_networks_b200 import GpfqError, QuantizedCNN, hostnet
from test_host_conv_groups import GroupedOracleEngine, grouped_cnn, grouped_oracle_conv

pytestmark = pytest.mark.gpu

# (kernel, strides, rate, padding, (n_img, H, W), C, F, groups, bits, alphabet scalar)
LAYERS = {
    "3x3_same_g8": ((3, 3), (1, 1), (1, 1), "SAME", (4, 12, 12), 32, 32, 8, 3, 3),             # Cg = Fg = 4, correlation form
    "3x3_stride2_cg4": ((3, 3), (2, 2), (1, 1), "SAME", (4, 13, 12), 8, 6, 2, 3, 3),           # Cg = 4, Fg = 3
    "1x1_g3": ((1, 1), (1, 1), (1, 1), "VALID", (4, 8, 9), 6, 9, 3, 2, 3),                     # Cg = 2, Fg = 3
    "7x7_groups_eq_c_fg1": ((7, 7), (1, 1), (1, 1), "SAME", (4, 10, 11), 6, 6, 6, 3, 3),        # depthwise, Fg = 1
    "7x7_groups_eq_c_fg2": ((7, 7), (1, 1), (1, 1), "SAME", (4, 10, 11), 5, 10, 5, 4, 4),       # depthwise, Fg = 2
    "5x5_rate22_cg3_fg5": ((5, 5), (1, 1), (2, 2), "SAME", (4, 12, 12), 6, 10, 2, 3, 3),
    "3x3_fg150": ((3, 3), (1, 1), (1, 1), "SAME", (3, 8, 9), 4, 300, 2, 3, 3),                  # Fg crosses the 128-thread block
    "5x3_fg150": ((5, 3), (1, 1), (1, 1), "SAME", (3, 8, 9), 4, 300, 2, 3, 3),                  # ... and the warp-per-filter walk
}


def _inputs(rng, n_img, H, Wd, C):
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    act[..., 0] = rng.standard_normal((n_img, H, Wd))
    actq[..., 0] = act[..., 0] + 0.05 * rng.standard_normal((n_img, H, Wd)).astype(np.float32)
    return act, actq


def _layer(name):
    ks, strides, rate, pad, (n_img, H, Wd), C, F, groups, bits, scalar = LAYERS[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    act, actq = _inputs(rng, n_img, H, Wd, C)
    W = (rng.uniform(-1, 1, (*ks, C // groups, F)) * 0.4).astype(np.float32)
    A = O.layer_alphabet(W, scalar, O.unit_alphabet(bits))
    return ks, dict(strides=strides, padding=pad, rate=rate), act, actq, W, A, groups


def _patches(act, actq, ks, geo):
    return lambda c: (O.channel_patches(act, c, ks, **geo), O.channel_patches(actq, c, ks, **geo))


def _mask(W, groups, c0, n_ch):
    """Entries of W that input channels c0 .. c0+n_ch-1 own."""
    Cg, Fg = W.shape[2], W.shape[3] // groups
    m = np.zeros(W.shape, bool)
    for c in range(c0, c0 + n_ch):
        m[:, :, c % Cg, (c // Cg) * Fg:(c // Cg + 1) * Fg] = True
    return m


def _crossing_shard(Cg, C):
    """A channel range that starts and ends inside groups and crosses at least one group boundary."""
    c0 = Cg // 2 if Cg > 1 else 1
    return c0, C - c0 - (Cg // 2 if Cg > 1 else 1)


@pytest.mark.parametrize("name", list(LAYERS))
def test_grouped_conv_matches_the_oracle(engine, name):
    import torch
    ks, geo, act, actq, W, A, groups = _layer(name)
    C, Cg, Fg = act.shape[-1], W.shape[2], W.shape[3] // groups
    kk = ks[0] * ks[1]
    td = lambda a: torch.from_numpy(a).cuda()
    for aq in (actq, None):                                   # hidden-layer and first-layer form
        src = act if aq is None else aq
        Q = engine.conv_layer_nhwc(act, aq, W, A, groups=groups, **geo)
        assert Q.shape == W.shape
        assert engine.last_stats["weights"] == kk * C * Fg
        assert O.agreement(Q, grouped_oracle_conv(W, groups, _patches(act, src, ks, geo), A)) == 1.0, aq is None
        # every other way into the same layer gives the same bits
        assert np.array_equal(engine.conv_layer_nhwc(td(act), None if aq is None else td(aq), td(W), A, groups=groups,
                                                     **geo).cpu().numpy(), Q)
        c0, n_ch = _crossing_shard(Cg, C)
        m = _mask(W, groups, c0, n_ch)
        assert m.any() and not m.all()
        for part in (engine.conv_layer_nhwc(act, aq, W, A, c0=c0, n_channels=n_ch, groups=groups, **geo),
                     engine.conv_layer_nhwc(td(act), None if aq is None else td(aq), td(W), A, c0=c0, n_channels=n_ch,
                                            groups=groups, **geo).cpu().numpy()):
            assert np.array_equal(part[m], Q[m]) and not part[~m].any()
        assert engine.last_stats["weights"] == kk * n_ch * Fg
        gram = engine.conv_gram_nhwc(act, aq, ks, **geo)
        assert np.array_equal(engine.conv_layer_from_gram(gram, W, A, groups=groups), Q)
        assert np.array_equal(engine.conv_layer_from_gram(gram, td(W), A, groups=groups).cpu().numpy(), Q)
        part = engine.conv_layer_from_gram(gram[c0:c0 + n_ch].contiguous(), W, A, c0=c0, n_channels=n_ch, groups=groups)
        assert np.array_equal(part[m], Q[m]) and not part[~m].any()


def test_grouped_conv_above_128_taps_takes_the_per_channel_path(engine):
    """13 x 11 (kk = 143) with groups 2: one Dense problem per input channel against its group's filters."""
    import torch
    rng = np.random.default_rng(143)
    ks, geo, groups = (13, 11), dict(strides=(1, 1), padding="SAME", rate=(1, 1)), 2
    act, actq = _inputs(rng, 2, 14, 13, 4)
    W = (rng.uniform(-1, 1, (*ks, 2, 6)) * 0.4).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(3))
    Q = engine.conv_layer_nhwc(act, actq, W, A, groups=groups, **geo)
    assert engine.last_stats["weights"] == 143 * 4 * 3
    assert O.agreement(Q, grouped_oracle_conv(W, groups, _patches(act, actq, ks, geo), A)) == 1.0
    td = lambda a: torch.from_numpy(a).cuda()
    assert np.array_equal(engine.conv_layer_nhwc(td(act), td(actq), td(W), A, groups=groups, **geo).cpu().numpy(), Q)
    m = _mask(W, groups, 1, 2)
    part = engine.conv_layer_nhwc(act, actq, W, A, c0=1, n_channels=2, groups=groups, **geo)
    assert np.array_equal(part[m], Q[m]) and not part[~m].any()


class _Groups1:
    """libgpfq with the ungrouped conv entry points answered by their grouped counterparts at groups = 1."""

    def __init__(self, lib):
        self._lib = lib

    def __getattr__(self, name):
        if name in ("gpfq_conv_layer_nhwc", "gpfq_conv_layer_from_gram"):
            fn = getattr(self._lib, name + "_grouped")
            return lambda *args: fn(*args, 1)
        return getattr(self._lib, name)


@pytest.mark.parametrize("ks,geo", [((3, 3), dict(strides=(1, 1), padding="SAME")),     # correlation form
                                    ((3, 3), dict(strides=(2, 1), padding="VALID")),    # im2col + kk = 9 walk
                                    ((5, 5), dict(strides=(1, 1), padding="SAME")),     # conv_gramx / conv_walkx
                                    ((13, 11), dict(strides=(1, 1), padding="SAME"))])  # per-channel path
def test_groups_1_through_the_grouped_symbols_is_the_ungrouped_call(engine, ks, geo):
    rng = np.random.default_rng(ks[0] * 31 + geo["strides"][0])
    act, actq = _inputs(rng, 4, 16, 14, 32)
    W = (rng.uniform(-1, 1, (*ks, 32, 5)) * 0.3).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(3))
    Q = engine.conv_layer_nhwc(act, actq, W, A, c0=3, n_channels=27, **geo)
    stats = dict(engine.last_stats)
    gram = engine.conv_gram_nhwc(act, actq, ks, **geo) if ks[0] * ks[1] <= 128 else None
    Qg = None if gram is None else engine.conv_layer_from_gram(gram, W, A)
    gstats = dict(engine.last_stats)
    lib = engine._lib
    engine._lib = _Groups1(lib)
    try:
        assert np.array_equal(engine.conv_layer_nhwc(act, actq, W, A, c0=3, n_channels=27, **geo), Q)
        assert engine.last_stats["kernel_launches"] == stats["kernel_launches"] and engine.last_stats["weights"] == stats["weights"]
        if gram is not None:
            assert np.array_equal(engine.conv_layer_from_gram(gram, W, A), Qg)
            assert engine.last_stats["kernel_launches"] == gstats["kernel_launches"]
    finally:
        engine._lib = lib


def test_grouped_walk_equals_per_group_calls_on_the_same_grams(engine):
    """One grouped walk over all channels equals `groups` ungrouped walks of the group slices (Grams of channels g Cg ..,
    kernel columns g Fg ..), bit for bit."""
    for name in ("3x3_same_g8", "5x5_rate22_cg3_fg5", "7x7_groups_eq_c_fg2"):
        ks, geo, act, actq, W, A, groups = _layer(name)
        Cg, Fg = W.shape[2], W.shape[3] // groups
        gram = engine.conv_gram_nhwc(act, actq, ks, **geo)
        Q = engine.conv_layer_from_gram(gram, W, A, groups=groups)
        ref = np.zeros(W.shape)
        for g in range(groups):
            Wg = np.ascontiguousarray(W[:, :, :, g * Fg:(g + 1) * Fg])
            ref[:, :, :, g * Fg:(g + 1) * Fg] = engine.conv_layer_from_gram(gram[g * Cg:(g + 1) * Cg].contiguous(), Wg, A)
        assert np.array_equal(Q, ref), name


def test_groups_equal_to_channels_is_a_depthwise_layer(engine):
    """Conv2D(groups=C, filters=C*M) equals DepthwiseConv2D(depth_multiplier=M) with its (kh, kw, C, M) kernel stored as
    (kh, kw, 1, C*M), bit for bit, in the engine and in the mirror."""
    rng = np.random.default_rng(9)
    C, M = 6, 3
    act, actq = _inputs(rng, 4, 11, 10, C)
    Wd = (rng.uniform(-1, 1, (7, 7, C, M)) * 0.4).astype(np.float32)
    A = O.layer_alphabet(Wd, 3, O.unit_alphabet(3))
    Qd = engine.conv_layer_nhwc(act, actq, Wd, A, padding="SAME")
    Qg = engine.conv_layer_nhwc(act, actq, Wd.reshape(7, 7, 1, C * M), A, padding="SAME", groups=C)
    assert np.array_equal(Qg.reshape(Qd.shape), Qd)
    # the same through QuantizedCNN: a network with a DepthwiseConv2D and its grouped twin
    L = hostnet
    x = rng.random((32, 12, 12, 3)).astype(np.float32)
    seq = hostnet.ArraySequence(x, np.zeros(32), 16)
    nd = L.Sequential([L.Conv2D(C, 3, padding="same", activation="relu"),
                       L.DepthwiseConv2D(5, padding="same", depth_multiplier=M, activation="relu"),
                       L.Flatten(), L.Dense(4, activation="softmax")], input_shape=(12, 12, 3), seed=2)
    ng = L.Sequential([L.Conv2D(C, 3, padding="same", activation="relu"),
                       L.Conv2D(C * M, 5, padding="same", groups=C, activation="relu"),
                       L.Flatten(), L.Dense(4, activation="softmax")], input_shape=(12, 12, 3), seed=2)
    w = nd.get_weights()
    ng.set_weights([w[0], w[1], w[2].reshape(5, 5, 1, C * M), w[3], w[4], w[5]])
    qd, qg = (QuantizedCNN(n, 16, seq, bits=3, alphabet_scalar=3) for n in (nd, ng))
    qd.quantize_network()
    qg.quantize_network()
    Kd, Kg = qd.quantized_net.layers[1].get_weights()[0], qg.quantized_net.layers[1].get_weights()[0]
    assert np.array_equal(Kg.reshape(Kd.shape), Kd)


def test_grouped_several_alphabets_in_one_call(engine):
    ks, geo, act, actq, W, A, groups = _layer("3x3_stride2_cg4")
    alphabets = [O.layer_alphabet(W, 2, O.unit_alphabet(np.log2(3))), O.layer_alphabet(W, 3, O.unit_alphabet(2)),
                 O.layer_alphabet(W, 5, O.unit_alphabet(6))]
    c0, n_ch = 2, 5
    m = _mask(W, groups, c0, n_ch)
    for aq in (actq, None):
        Qm = engine.conv_layer_nhwc(act, aq, W, alphabets, c0=c0, n_channels=n_ch, groups=groups, **geo)
        assert Qm.shape == (3, *W.shape)
        for a, Aa in enumerate(alphabets):
            single = engine.conv_layer_nhwc(act, aq, W, Aa, c0=c0, n_channels=n_ch, groups=groups, **geo)
            assert np.array_equal(Qm[a], single), a
            assert not Qm[a][~m].any(), a
            ref = grouped_oracle_conv(W, groups, _patches(act, act if aq is None else aq, ks, geo), Aa, c0, n_ch)
            assert O.agreement(Qm[a], ref) == 1.0, a


def test_bad_groups_raise(engine, monkeypatch):
    import torch
    rng = np.random.default_rng(1)
    act, actq = _inputs(rng, 2, 6, 6, 8)
    W = (rng.uniform(-1, 1, (3, 3, 2, 6)) * 0.4).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(3))
    with pytest.raises(ValueError):
        engine.conv_layer_nhwc(act, actq, W, A, groups=3)               # 2 * 3 != 8 input channels
    with pytest.raises(ValueError):
        engine.conv_layer_nhwc(act, actq, W, A)                         # a grouped kernel without groups
    with pytest.raises(ValueError):
        engine.conv_layer_nhwc(act, actq, (rng.uniform(-1, 1, (3, 3, 2, 5))).astype(np.float32), A, groups=4)   # F = 5
    with pytest.raises(ValueError):
        engine.conv_layer_from_gram(torch.zeros((8, 2, 9, 9), dtype=torch.float64, device="cuda"), W, A, groups=0)
    # the library checks them too
    monkeypatch.setattr(type(engine), "_check_groups", staticmethod(lambda g, C, Cg, F: int(g)))
    with pytest.raises(GpfqError):
        engine.conv_layer_nhwc(act, actq, (rng.uniform(-1, 1, (3, 3, 3, 6))).astype(np.float32), A, groups=3)   # 8 % 3
    with pytest.raises(GpfqError):
        engine.conv_layer_nhwc(act, actq, (rng.uniform(-1, 1, (3, 3, 2, 6))).astype(np.float32), A, groups=4)   # 6 % 4
    # straight through the C ABI: a (3, 3, 2, 8) kernel with 8 filters, Grams of 8 channels
    gram = engine.conv_gram_nhwc(act, actq, (3, 3))
    Wd = torch.from_numpy((rng.uniform(-1, 1, (3, 3, 2, 8)) * 0.4).astype(np.float32)).cuda()
    K = np.array([len(A)], np.int32)
    Q = torch.zeros((3, 3, 2, 8), dtype=torch.float64, device="cuda")
    for groups, C, want in ((4, 8, 0), (0, 8, 1), (-4, 8, 1), (3, 8, 1), (3, 9, 1), (16, 16, 1)):   # C % groups, F % groups
        rc = engine._lib.gpfq_conv_layer_from_gram_grouped(engine._ctx, c_void_p(gram.data_ptr()), 9, c_void_p(Wd.data_ptr()), C,
                                                          8, 0, min(C, 8), A.ctypes.data_as(POINTER(c_double)),
                                                          K.ctypes.data_as(POINTER(c_int32)), 1, c_void_p(Q.data_ptr()), 7, None,
                                                          groups)
        assert rc == want, (groups, C, rc)


@pytest.mark.parametrize("conv_path", ["nhwc", "patches"])
def test_cnn_with_grouped_layers_matches_the_oracle_walk(conv_path):
    from test_gpu_network import _compare
    rng = np.random.default_rng(31)
    net = grouped_cnn(seed=6)
    x = rng.random((48, 14, 14, 3)).astype(np.float32)
    seq = hostnet.ArraySequence(x, rng.integers(0, 10, 48), 16)
    qg = QuantizedCNN(net, 16, seq, bits=3, alphabet_scalar=3, conv_path=conv_path)
    qg.quantize_network()
    qo = QuantizedCNN(net, 16, seq, bits=3, alphabet_scalar=3)
    qo.__class__ = type("GroupedOracleQuantizedCNN", (QuantizedCNN,), {"engine": property(lambda self: GroupedOracleEngine())})
    qo.quantize_network()
    _compare(qg, qo, x[:32], {"Dense", "Conv2D"})


def test_grid_runner_with_grouped_layers_matches_point_by_point_runs():
    from quantized_neural_networks_b200 import QuantizedCNNGrid
    rng = np.random.default_rng(32)
    net = grouped_cnn(seed=7)
    x = rng.random((48, 14, 14, 3)).astype(np.float32)
    seq = hostnet.ArraySequence(x, rng.integers(0, 10, 48), 16)
    quiet = type("L", (), {"info": staticmethod(lambda m: None)})()
    bits_list, scalars = [np.log2(3), 3], [2, 4]
    grid = QuantizedCNNGrid(net, 16, seq, bits_list, scalars, logger=quiet).quantize_network()
    for (b, c), qnet in zip(grid.grid, grid.quantized_nets):
        single = QuantizedCNN(net, 16, seq, logger=quiet, bits=b, alphabet_scalar=c)
        single.quantize_network()
        for idx, layer in enumerate(net.layers):
            if layer.__class__.__name__ in ("Dense", "Conv2D"):
                Wg, Ws = qnet.layers[idx].get_weights()[0], single.quantized_net.layers[idx].get_weights()[0]
                assert float(np.mean(Wg == Ws)) >= 0.9999, (b, c, idx)
                assert not np.array_equal(Wg, layer.get_weights()[0])
        assert np.array_equal(qnet.predict(x[:32]).argmax(-1), single.quantized_net.predict(x[:32]).argmax(-1))
