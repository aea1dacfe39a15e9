"""GPU: conv kernels of any size up to 128 taps (5 x 5, 7 x 7 / 2, 11 x 11 / 4, 1 x 7, 7 x 1, 8 x 16, ...) through the batched
Gram and walk kernels for a runtime kh * kw (conv_gramx_kernel / conv_walkx_kernel), with the Gram-only pair of the image
split; kernels above 128 taps through the one-Dense-problem-per-channel path.

The checkers are those of test_gpu_conv_geometry.py: fp64 NumPy Grams of the oracle's patch matrices (`O.channel_patches`)
within 1e-12 |Xq| |X|^T, and the literal C oracle walk for the quantized kernel, entry for entry.
"""
import numpy as np
import pytest

from oracle import c_oracle, gpfq_oracle as O
from quantized_neural_networks_b200 import GpfqError, QuantizedCNN, hostnet
from quantized_neural_networks_b200.engine import CONV_SUPPORTED_KK

pytestmark = pytest.mark.gpu

# (kernel, strides, rate, padding, (n_img, H, W), C, F, bits, alphabet scalar)
LAYERS = {
    "5x5_same": ((5, 5), (1, 1), (1, 1), "SAME", (4, 12, 11), 3, 6, 3, 3),
    "5x5_stride2_valid": ((5, 5), (2, 2), (1, 1), "VALID", (5, 13, 12), 3, 5, np.log2(3), 2),
    "7x7_stride2_same_c3": ((7, 7), (2, 2), (1, 1), "SAME", (4, 16, 15), 3, 8, 4, 4),
    "11x11_stride4_valid": ((11, 11), (4, 4), (1, 1), "VALID", (3, 31, 27), 3, 6, 3, 3),        # n = 90
    "1x7_same": ((1, 7), (1, 1), (1, 1), "SAME", (4, 9, 13), 4, 5, 3, 3),
    "7x1_same": ((7, 1), (1, 1), (1, 1), "SAME", (4, 13, 9), 4, 5, 3, 3),
    "3x5_rate21_same": ((3, 5), (1, 1), (2, 1), "SAME", (4, 10, 11), 3, 4, 2, 3),
    "4x4_rate12_same": ((4, 4), (1, 1), (1, 2), "SAME", (4, 10, 12), 3, 4, 3, 3),               # kk = 16
    "5x5_rate33_dead_taps": ((5, 5), (1, 1), (3, 3), "SAME", (6, 5, 5), 3, 4, 3, 3),
    "8x16_kk128": ((8, 16), (1, 1), (1, 1), "SAME", (2, 10, 18), 3, 4, 3, 3),                   # the limit
    "5x3_F150": ((5, 3), (1, 1), (1, 1), "SAME", (3, 8, 9), 3, 150, 3, 3),                      # more than 128 filters
    "5x5_depthwise_F1": ((5, 5), (1, 1), (1, 1), "SAME", (4, 10, 10), 6, 1, 3, 3),              # one filter per channel
}


def _inputs(rng, n_img, H, Wd, C):
    """ReLU activations and a perturbed twin; channel 0 signed, channel 1 zero except on the bottom row."""
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    act[..., 0] = rng.standard_normal((n_img, H, Wd))
    actq[..., 0] = act[..., 0] + 0.05 * rng.standard_normal((n_img, H, Wd)).astype(np.float32)
    act[:, :-1, :, 1] = 0
    actq[:, :-1, :, 1] = 0
    return act, actq


def _assert_grams(gram, pats, same=False):
    """Lower triangle + diagonal of G1 = Xq X^T and G2 = Xq Xq^T within 1e-12 of |Xq| |X|^T entrywise; G1 == G2 in the
    first-layer form."""
    gram = gram.cpu().numpy()
    kk = gram.shape[-1]
    tri = np.tril_indices(kk)
    for c, (Xp, Xqp) in enumerate(pats):
        x, q = Xp.astype(np.float64), Xqp.astype(np.float64)
        for G, R, S in ((gram[c, 0], q @ x.T, np.abs(q) @ np.abs(x).T), (gram[c, 1], q @ q.T, np.abs(q) @ np.abs(q).T)):
            err = np.abs(G[tri] - R[tri])
            assert np.all(err <= 1e-12 * S[tri]), (c, float(np.max(err / np.maximum(S[tri], 1e-300))))
        if same:
            assert np.array_equal(gram[c, 0][tri], gram[c, 1][tri]), c


def _layer(name):
    ks, strides, rate, pad, (n_img, H, Wd), C, F, bits, scalar = LAYERS[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    act, actq = _inputs(rng, n_img, H, Wd, C)
    W = (rng.uniform(-1, 1, (*ks, C, F)) * 0.4).astype(np.float32)
    A = O.layer_alphabet(W, scalar, O.unit_alphabet(bits))
    return ks, dict(strides=strides, padding=pad, rate=rate), act, actq, W, A


@pytest.mark.parametrize("name", list(LAYERS))
def test_conv_any_kernel_matches_the_oracle(engine, name):
    import torch
    ks, geo, act, actq, W, A = _layer(name)
    C = act.shape[-1]
    assert ks[0] * ks[1] in CONV_SUPPORTED_KK
    pats = [(O.channel_patches(act, c, ks, **geo), O.channel_patches(actq, c, ks, **geo)) for c in range(C)]
    first = [(O.channel_patches(act, c, ks, **geo),) * 2 for c in range(C)]

    # 1. the Gram stage alone, summed over two image halves
    half = act.shape[0] // 2
    gram = engine.conv_gram_nhwc(act[:half], actq[:half], ks, **geo) + engine.conv_gram_nhwc(act[half:], actq[half:], ks, **geo)
    _assert_grams(gram, pats)
    gram1 = engine.conv_gram_nhwc(act[:half], None, ks, **geo) + engine.conv_gram_nhwc(act[half:], None, ks, **geo)
    _assert_grams(gram1, first, same=True)

    # 2. the quantized kernel against the literal oracle walk, hidden-layer and first-layer form
    Q = engine.conv_layer_nhwc(act, actq, W, A, **geo)
    assert O.agreement(Q, c_oracle.quantize_conv_layer(W, lambda c: pats[c], A)) == 1.0
    Q1 = engine.conv_layer_nhwc(act, None, W, A, **geo)
    assert O.agreement(Q1, c_oracle.quantize_conv_layer(W, lambda c: first[c], A)) == 1.0
    if name == "5x5_rate33_dead_taps":
        # on 5 x 5 images with pad 6 a tap (r, s) reads pixel (i + 3 r - 6, j + 3 s - 6): only r, s in {1, 2, 3} see the image
        live = np.zeros((5, 5), bool)
        live[1:4, 1:4] = True
        assert not Q[~live].any() and not Q1[~live].any() and Q[live].any()
        g = gram.cpu().numpy()
        dead = np.flatnonzero(~live.ravel())
        assert not g[:, 1][:, dead, :].any() and not g[:, 1][:, :, dead].any()

    # 3. every other way into the same layer gives the same bits
    td = lambda a: torch.from_numpy(a).cuda()
    assert np.array_equal(engine.conv_layer_nhwc(td(act), td(actq), td(W), A, **geo).cpu().numpy(), Q)
    part = engine.conv_layer_nhwc(act, actq, W, A, c0=1, n_channels=C - 1, **geo)
    assert np.array_equal(part[:, :, 1:], Q[:, :, 1:]) and not part[:, :, 0].any()
    assert np.array_equal(engine.conv_channels([p[0] for p in pats], [p[1] for p in pats], W, A), Q)
    assert np.array_equal(engine.conv_channels([p[0] for p in first], None, W, A), Q1)
    assert np.array_equal(engine.conv_layer_from_gram(gram, W, A), Q)
    assert np.array_equal(engine.conv_layer_from_gram(gram1, W, A), Q1)


@pytest.mark.parametrize("ks", [(5, 5), (1, 7), (8, 16)])
def test_conv_any_kernel_is_one_batched_call(engine, ks):
    """The whole layer is one batched call: the kernel launches do not grow with the channel count (the per-channel path
    ran one Dense problem, i.e. several launches, per channel)."""
    rng = np.random.default_rng(3)
    launches = {}
    for C in (2, 16):
        act, actq = _inputs(rng, 3, 9, 10, C)
        W = (rng.uniform(-1, 1, (*ks, C, 4)) * 0.4).astype(np.float32)
        A = O.layer_alphabet(W, 3, O.unit_alphabet(3))
        engine.conv_layer_nhwc(act, actq, W, A)
        n_nhwc = engine.last_stats["kernel_launches"]
        pats = [O.channel_patches(act, c, ks, padding="SAME") for c in range(C)]
        engine.conv_channels(pats, None, W, A)
        launches[C] = (n_nhwc, engine.last_stats["kernel_launches"])
    assert launches[2] == launches[16] and min(launches[2]) > 0, launches


def test_conv_any_kernel_several_alphabets_in_one_call(engine):
    """Ternary, 2-bit and 6-bit (64 levels) alphabets batched in one call through a 7 x 7 layer with a channel shard: each
    alphabet's block equals its single-alphabet call and the oracle."""
    rng = np.random.default_rng(77)
    ks, strides, pad = (7, 7), (1, 2), "SAME"
    act, actq = _inputs(rng, 5, 11, 12, 4)
    C, F = 4, 5
    W = (rng.uniform(-1, 1, (*ks, C, F)) * 0.4).astype(np.float32)
    alphabets = [O.layer_alphabet(W, 2, O.unit_alphabet(np.log2(3))), O.layer_alphabet(W, 3, O.unit_alphabet(2)),
                 O.layer_alphabet(W, 5, O.unit_alphabet(6))]
    assert len(alphabets[2]) == 64
    for aq in (actq, None):
        src = act if aq is None else aq
        pats = [(O.channel_patches(act, c, ks, strides, pad), O.channel_patches(src, c, ks, strides, pad)) for c in range(C)]
        Qm = engine.conv_layer_nhwc(act, aq, W, alphabets, strides=strides, padding=pad, c0=1, n_channels=C - 1)
        assert Qm.shape == (3, *ks, C, F)
        for a, A in enumerate(alphabets):
            single = engine.conv_layer_nhwc(act, aq, W, A, strides=strides, padding=pad, c0=1, n_channels=C - 1)
            assert np.array_equal(Qm[a], single), a
            assert not Qm[a][:, :, 0].any(), a
            Qref = c_oracle.quantize_conv_layer(W, lambda c: pats[c], A)
            assert O.agreement(Qm[a][:, :, 1:], Qref[:, :, 1:]) == 1.0, a


def test_conv_any_kernel_host_image_chunks(engine):
    """Host activations above the 96 MB staging target (44 x 160 x 160 x 24 fp32, 108 MB) through a 5 x 5 / 4 layer: image chunks
    of 40 and 4 images, each with its own partial slots.  Same quantized kernel as the device-tensor call and as the oracle;
    both Grams within the fp64 bound of NumPy's (the two calls associate their partial sums differently)."""
    import torch
    rng = np.random.default_rng(55)
    n_img, H, Wd, C, F = 44, 160, 160, 24, 2
    ks, geo = (5, 5), dict(strides=(4, 4), padding="SAME", rate=(1, 1))
    act, actq = _inputs(rng, n_img, H, Wd, C)
    W = (rng.uniform(-1, 1, (*ks, C, F)) * 0.3).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(np.log2(3)))
    pats = [(O.channel_patches(act, c, ks, **geo), O.channel_patches(actq, c, ks, **geo)) for c in range(C)]
    Q = engine.conv_layer_nhwc(act, actq, W, A, **geo)
    Qd = engine.conv_layer_nhwc(torch.from_numpy(act).cuda(), torch.from_numpy(actq).cuda(), torch.from_numpy(W).cuda(), A, **geo)
    assert np.array_equal(Qd.cpu().numpy(), Q)
    assert O.agreement(Q, c_oracle.quantize_conv_layer(W, lambda c: pats[c], A)) == 1.0
    gram = engine.conv_gram_nhwc(act, actq, ks, **geo)
    gram_d = engine.conv_gram_nhwc(torch.from_numpy(act).cuda(), torch.from_numpy(actq).cuda(), ks, **geo)
    _assert_grams(gram, pats)
    _assert_grams(gram_d, pats)
    assert np.array_equal(engine.conv_layer_from_gram(gram, W, A), Q)


def test_conv_kk128_with_512_channels(engine):
    """kk = 128 (8 x 16) with 512 channels: 256 KB of partial Gram per channel and slot, 128 MB per slot of all channels.  The
    partial workspace stays within 1 GiB although the shapes ask for more slots: device activations with 10368 patch columns
    per channel would take 9 column chunks (capped to 8), and 906 MB of host activations in 96 MB image chunks would take 9
    image chunks of 18 column chunks each (capped to 8 image chunks of one).  Both calls succeed, and a sample of channels
    equals the oracle and the NumPy Grams."""
    import torch
    ks, geo = (8, 16), dict(strides=(1, 1), padding="SAME", rate=(1, 1))
    C, F, sample = 512, 2, [0, 1, 255, 511]
    limit = 1 << 30
    # device activations: the column chunks are capped
    rng = np.random.default_rng(128)
    act, actq = _inputs(rng, 8, 36, 36, C)
    W = (rng.uniform(-1, 1, (*ks, C, F)) * 0.4).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(3))
    td = lambda a: torch.from_numpy(a).cuda()
    Q = engine.conv_layer_nhwc(td(act), td(actq), td(W), A, **geo).cpu().numpy()
    assert limit // 2 < engine.conv_partial_bytes() <= limit, engine.conv_partial_bytes()
    pats = {c: (O.channel_patches(act, c, ks, **geo), O.channel_patches(actq, c, ks, **geo)) for c in sample}
    Qref = c_oracle.quantize_conv_layer(np.ascontiguousarray(W[:, :, sample]), lambda i: pats[sample[i]], A)
    assert O.agreement(Q[:, :, sample], Qref) == 1.0
    gram = engine.conv_gram_nhwc(td(act), td(actq), ks, **geo)
    assert engine.conv_partial_bytes() <= limit
    _assert_grams(gram[sample], [pats[c] for c in sample])
    assert np.array_equal(engine.conv_layer_from_gram(gram, W, A), Q)
    del act, actq, pats, gram

    # host activations (first-layer form) above eight 96 MB staging chunks: the image chunks are capped
    rng = np.random.default_rng(129)
    act = np.maximum(rng.standard_normal((1728, 16, 16, C), dtype=np.float32), 0)
    Q1 = engine.conv_layer_nhwc(act, None, W, A, **geo)
    assert limit // 2 < engine.conv_partial_bytes() <= limit, engine.conv_partial_bytes()
    first = {c: (O.channel_patches(act, c, ks, **geo),) * 2 for c in sample[:2]}
    Qref1 = c_oracle.quantize_conv_layer(np.ascontiguousarray(W[:, :, sample[:2]]), lambda i: first[sample[i]], A)
    assert O.agreement(Q1[:, :, sample[:2]], Qref1) == 1.0


def test_conv_above_128_taps_takes_the_per_channel_path(engine):
    """13 x 11 (kk = 143) still quantizes, one Dense problem per channel, equal to the oracle; it has no Gram-only pair."""
    import torch
    rng = np.random.default_rng(143)
    ks, geo = (13, 11), dict(strides=(1, 1), padding="SAME", rate=(1, 1))
    act, actq = _inputs(rng, 2, 14, 13, 3)
    W = (rng.uniform(-1, 1, (*ks, 3, 4)) * 0.4).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(3))
    assert 143 not in CONV_SUPPORTED_KK
    pats = [(O.channel_patches(act, c, ks, **geo), O.channel_patches(actq, c, ks, **geo)) for c in range(3)]
    Q = engine.conv_layer_nhwc(act, actq, W, A, **geo)
    assert O.agreement(Q, c_oracle.quantize_conv_layer(W, lambda c: pats[c], A)) == 1.0
    with pytest.raises(GpfqError):
        engine.conv_gram_nhwc(act, actq, ks, **geo)
    with pytest.raises(GpfqError):
        engine.conv_layer_from_gram(torch.zeros((3, 2, 143, 143), dtype=torch.float64, device="cuda"), W, A)


@pytest.mark.parametrize("conv_path", ["nhwc", "patches"])
def test_cnn_with_large_kernels_matches_the_oracle_walk(conv_path):
    """A small network with 11 x 11 / 4, 5 x 5, 7 x 1, 1 x 7 and a 5 x 5 DepthwiseConv2D, through both conv paths, against
    the same walk with the hot path replaced by the oracle (test_gpu_network.py)."""
    from test_gpu_network import _compare, _with_oracle
    rng = np.random.default_rng(21)
    L = hostnet
    net = L.Sequential([L.Conv2D(8, 11, strides=4, padding="valid", activation="relu"),
                        L.Conv2D(8, 5, padding="same", activation="relu"),
                        L.Conv2D(6, (7, 1), padding="same", activation="relu"),
                        L.Conv2D(6, (1, 7), padding="same", activation="relu"),
                        L.DepthwiseConv2D(5, padding="same", activation="relu"),
                        L.Flatten(), L.Dense(10, activation="softmax")], input_shape=(35, 35, 3), seed=6)
    x = rng.random((48, 35, 35, 3)).astype(np.float32)
    seq = hostnet.ArraySequence(x, rng.integers(0, 10, 48), 16)
    qg = QuantizedCNN(net, 16, seq, bits=3, alphabet_scalar=3, conv_path=conv_path)
    qg.quantize_network()
    qo = _with_oracle(QuantizedCNN, net, 16, seq, bits=3, alphabet_scalar=3)
    qo.quantize_network()
    _compare(qg, qo, x[:32], {"Dense", "Conv2D", "DepthwiseConv2D"})
