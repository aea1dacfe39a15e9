"""GPU: conv layers of every geometry the reference accepts (quantized_network.py:686-727, tf.image.extract_patches :158-172),
not just the square 3 x 3 / stride 1 kernels of VGG16 and the CIFAR10 CNN: non-square kernels (every kh * kw with its own Gram
and walk kernels, and sizes without), asymmetric strides, strides beyond the kernel extent, dilation on either axis, SAME
padding with a nonzero top / left pad, VALID outputs one pixel high or wide, more than 128 filters, and host activations
above one staging chunk.

The checkers: fp64 NumPy Grams of the oracle's patch matrices (`O.channel_patches`, pinned to hostnet and torch's unfold in
test_host.py) for the Gram stage, and the literal C oracle walk for the quantized kernel, which must agree entry for entry.
Every other way into the same layer (device tensors, channel shards, patch matrices, the Gram-only pair) gives the same bits.
"""
import numpy as np
import pytest

from oracle import c_oracle, gpfq_oracle as O
from quantized_neural_networks_b200 import GpfqError
from quantized_neural_networks_b200.engine import CONV_SUPPORTED_KK

pytestmark = pytest.mark.gpu

# (kernel, strides, rate, padding, (n_img, H, W), C, F, bits, alphabet scalar)
LAYERS = {
    "1x2_stride13_same": ((1, 2), (1, 3), (1, 1), "SAME", (6, 9, 11), 3, 5, np.log2(3), 2),       # stride > extent
    "2x1_rate21_valid": ((2, 1), (1, 1), (2, 1), "VALID", (5, 8, 7), 3, 4, 3, 3),
    "1x3_stride21_same": ((1, 3), (2, 1), (1, 1), "SAME", (4, 9, 10), 4, 6, 4, 4),                # left pad 1
    "3x1_rate21_same": ((3, 1), (1, 1), (2, 1), "SAME", (5, 9, 6), 3, 3, 2, 3),                    # top pad 2
    "3x1_stride12_valid_ho1": ((3, 1), (1, 2), (1, 1), "VALID", (12, 3, 8), 3, 4, np.log2(3), 2),
    "1x4_rate12_same": ((1, 4), (1, 1), (1, 2), "SAME", (40, 12, 13), 3, 5, 3, 3),                 # left pad 3, two chunks
    "4x1_stride31_valid": ((4, 1), (3, 1), (1, 1), "VALID", (6, 13, 5), 3, 4, 4, 4),
    "2x3_rate23_valid_wo1": ((2, 3), (1, 1), (2, 3), "VALID", (7, 8, 7), 3, 5, np.log2(3), 3),
    "3x2_stride22_same_F150": ((3, 2), (2, 2), (1, 1), "SAME", (4, 9, 9), 3, 150, 3, 3),           # two filter blocks
    "1x6_same": ((1, 6), (1, 1), (1, 1), "SAME", (3, 5, 12), 3, 4, 2, 2),
    "1x9_same": ((1, 9), (1, 1), (1, 1), "SAME", (4, 6, 15), 3, 4, 4, 4),                          # n % 4 == 0
    "9x1_valid_ho1": ((9, 1), (1, 1), (1, 1), "VALID", (5, 9, 7), 3, 4, 3, 3),                     # n = 35
    "3x3_stride12_same": ((3, 3), (1, 2), (1, 1), "SAME", (4, 11, 12), 4, 5, np.log2(3), 2),
    "3x3_rate22_same": ((3, 3), (1, 1), (2, 2), "SAME", (3, 10, 9), 3, 4, 3, 3),                   # n = 270
    "3x3_rate44_dead_taps": ((3, 3), (1, 1), (4, 4), "SAME", (6, 4, 4), 3, 4, 3, 3),
    "1x1_stride32_valid": ((1, 1), (3, 2), (1, 1), "VALID", (4, 10, 9), 3, 4, 3, 3),               # stride > extent
    "1x5_rate12_same": ((1, 5), (1, 1), (1, 2), "SAME", (4, 7, 11), 3, 4, 3, 3),                   # no own kernel
    "2x5_stride21_valid": ((2, 5), (2, 1), (1, 1), "VALID", (5, 9, 8), 3, 4, np.log2(3), 2),       # no own kernel
}


def _inputs(rng, n_img, H, Wd, C):
    """ReLU activations and a perturbed twin; channel 0 signed (Gram entries with cancellation), channel 1 zero except on the
    bottom row (taps that never reach it are dead directions)."""
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    act[..., 0] = rng.standard_normal((n_img, H, Wd))
    actq[..., 0] = act[..., 0] + 0.05 * rng.standard_normal((n_img, H, Wd)).astype(np.float32)
    act[:, :-1, :, 1] = 0
    actq[:, :-1, :, 1] = 0
    return act, actq


def _assert_grams(gram, pats, same=False):
    """gram: (C, 2, kk, kk) from conv_gram_nhwc; pats[c] = (Xp, Xqp).  Lower triangle + diagonal of G1 = Xq X^T and
    G2 = Xq Xq^T within 1e-12 of |Xq| |X|^T entrywise (dead entries exactly 0); the first-layer form has G1 == G2."""
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


class _option:
    def __init__(self, engine, key, value):
        self.engine, self.key, self.value = engine, key, value

    def __enter__(self):
        self.engine.set_option(self.key, self.value)

    def __exit__(self, *exc):
        self.engine.set_option(self.key, 0)


@pytest.mark.parametrize("name", list(LAYERS))
def test_conv_geometry_matches_the_oracle(engine, name):
    import torch
    ks, strides, rate, pad, (n_img, H, Wd), C, F, bits, scalar = LAYERS[name]
    kk = ks[0] * ks[1]
    rng = np.random.default_rng(sum(map(ord, name)))
    act, actq = _inputs(rng, n_img, H, Wd, C)
    W = (rng.uniform(-1, 1, (*ks, C, F)) * 0.4).astype(np.float32)
    A = O.layer_alphabet(W, scalar, O.unit_alphabet(bits))
    geo = dict(strides=strides, padding=pad, rate=rate)
    pats = [(O.channel_patches(act, c, ks, strides, pad, rate), O.channel_patches(actq, c, ks, strides, pad, rate))
            for c in range(C)]
    first = [(O.channel_patches(act, c, ks, strides, pad, rate),) * 2 for c in range(C)]

    # 1. the Gram stage alone, summed over two image chunks (what the ranks of an image-split job all-reduce)
    half = n_img // 2
    if kk in CONV_SUPPORTED_KK:
        gram = engine.conv_gram_nhwc(act[:half], actq[:half], ks, **geo) + engine.conv_gram_nhwc(act[half:], actq[half:], ks, **geo)
        _assert_grams(gram, pats)
        gram1 = engine.conv_gram_nhwc(act[:half], None, ks, **geo) + engine.conv_gram_nhwc(act[half:], None, ks, **geo)
        _assert_grams(gram1, first, same=True)
    else:
        with pytest.raises(GpfqError):
            engine.conv_gram_nhwc(act, actq, ks, **geo)

    # 2. the quantized kernel against the literal oracle walk, hidden-layer and first-layer form
    Q = engine.conv_layer_nhwc(act, actq, W, A, **geo)
    assert O.agreement(Q, c_oracle.quantize_conv_layer(W, lambda c: pats[c], A)) == 1.0
    Q1 = engine.conv_layer_nhwc(act, None, W, A, **geo)
    assert O.agreement(Q1, c_oracle.quantize_conv_layer(W, lambda c: first[c], A)) == 1.0
    if name == "3x3_rate44_dead_taps":
        # on 4 x 4 images with pad 4 a tap reads pixel (i + 4 r - 4, j + 4 s - 4): only the centre tap ever sees the image
        live = np.zeros((3, 3), bool)
        live[1, 1] = True
        assert not Q[~live].any() and not Q1[~live].any() and Q[live].any()

    # 3. every other way into the same layer gives the same bits
    td = lambda a: torch.from_numpy(a).cuda()
    assert np.array_equal(engine.conv_layer_nhwc(td(act), td(actq), td(W), A, **geo).cpu().numpy(), Q)
    part = engine.conv_layer_nhwc(act, actq, W, A, c0=1, n_channels=C - 1, **geo)
    assert np.array_equal(part[:, :, 1:], Q[:, :, 1:]) and not part[:, :, 0].any()
    assert np.array_equal(engine.conv_channels([p[0] for p in pats], [p[1] for p in pats], W, A), Q)
    assert np.array_equal(engine.conv_channels([p[0] for p in first], None, W, A), Q1)
    if kk in CONV_SUPPORTED_KK:
        assert np.array_equal(engine.conv_layer_from_gram(gram, W, A), Q)
        assert np.array_equal(engine.conv_layer_from_gram(gram1, W, A), Q1)

    # kk = 9 off the 3 x 3 / stride 1 planner goes through im2col + patch Grams: the TMA-staged (0), direct LDG (1) and
    # generic (2) kernels; all three fall back to the generic kernel when n % 4 != 0
    if kk == 9:
        for variant in (1, 2):
            with _option(engine, "conv_kernel", variant):
                assert np.array_equal(engine.conv_layer_nhwc(act, actq, W, A, **geo), Q), variant
                assert np.array_equal(engine.conv_layer_nhwc(act, None, W, A, **geo), Q1), variant
                _assert_grams(engine.conv_gram_nhwc(act, actq, ks, **geo), pats)


def test_conv_kernel_sizes_with_a_gram_only_path_are_the_engine_constant(engine):
    """CONV_SUPPORTED_KK (what the multi-GPU conv path reads to pick the image split) is the set the library serves: kernels
    (1, k), k = 1..10, have the Gram-only and from-Gram entry points exactly when k is in it."""
    import torch
    rng = np.random.default_rng(2)
    act = np.maximum(rng.standard_normal((2, 6, 12, 2)), 0).astype(np.float32)
    for k in range(1, 11):
        W = np.ones((1, k, 2, 3), np.float32)
        A = np.array([-1.0, 0.0, 1.0])
        if k in CONV_SUPPORTED_KK:
            gram = engine.conv_gram_nhwc(act, None, (1, k))
            assert gram.shape == (2, 2, k, k)
            engine.conv_layer_from_gram(gram, W, A)
        else:
            with pytest.raises(GpfqError):
                engine.conv_gram_nhwc(act, None, (1, k))
            with pytest.raises(GpfqError):
                engine.conv_layer_from_gram(torch.zeros((2, 2, k, k), dtype=torch.float64, device="cuda"), W, A)


@pytest.mark.parametrize("ks,strides,rate,pad", [((2, 3), (1, 2), (2, 1), "SAME"), ((1, 5), (2, 1), (1, 1), "VALID")])
def test_conv_several_alphabets_in_one_call(engine, ks, strides, rate, pad):
    """Alphabets batched in one call (the grid runner does this at the first layer) with a channel shard: each alphabet's
    output is its own (kh, kw, C, F) block, equal to its single-alphabet call and to the oracle -- through the kk = 6 walk
    kernel and through the one-Dense-problem-per-channel path of a size without its own kernel."""
    rng = np.random.default_rng(ks[0] * 10 + ks[1])
    n_img, H, Wd, C, F = 6, 9, 10, 4, 5
    act, actq = _inputs(rng, n_img, H, Wd, C)
    W = (rng.uniform(-1, 1, (*ks, C, F)) * 0.4).astype(np.float32)
    alphabets = [O.layer_alphabet(W, 2, O.unit_alphabet(np.log2(3))), O.layer_alphabet(W, 4, O.unit_alphabet(4)),
                 O.layer_alphabet(W, 3, O.unit_alphabet(2))]
    geo = dict(strides=strides, padding=pad, rate=rate)
    for aq in (actq, None):
        src = act if aq is None else aq
        pats = [(O.channel_patches(act, c, ks, strides, pad, rate), O.channel_patches(src, c, ks, strides, pad, rate))
                for c in range(C)]
        Qm = engine.conv_layer_nhwc(act, aq, W, alphabets, c0=1, n_channels=C - 1, **geo)
        assert Qm.shape == (3, *ks, C, F)
        for a, A in enumerate(alphabets):
            single = engine.conv_layer_nhwc(act, aq, W, A, c0=1, n_channels=C - 1, **geo)
            assert np.array_equal(Qm[a], single), a
            assert not Qm[a][:, :, 0].any(), a
            Qref = c_oracle.quantize_conv_layer(W, lambda c: pats[c], A)
            assert O.agreement(Qm[a][:, :, 1:], Qref[:, :, 1:]) == 1.0, a


def test_conv_patch_path_host_image_chunks(engine):
    """Host activations above the 96 MB staging target (44 x 128 x 128 x 40 fp32, 115 MB): a strided 3 x 3 layer goes through
    im2col + patch Grams in image chunks of 40 and 4 images, each with its own partial slots (the short last chunk leaves
    slots unused).  Same quantized kernel as the device-tensor call (one chunk), as the walk from the Gram-only call and as
    the oracle; Grams of both calls within the fp64 bound of NumPy's."""
    import torch
    from quantized_neural_networks_b200 import hostnet
    rng = np.random.default_rng(44)
    n_img, H, Wd, C, F = 44, 128, 128, 40, 2
    act, actq = _inputs(rng, n_img, H, Wd, C)
    W = (rng.uniform(-1, 1, (3, 3, C, F)) * 0.3).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(np.log2(3)))
    geo = dict(strides=(2, 2), padding="SAME", rate=(1, 1))

    def patches(a):   # hostnet.extract_patches of all channels at once: (C, 9, n_img * 64 * 64)
        p = hostnet.extract_patches(a, [1, 3, 3, 1], [1, 2, 2, 1], [1, 1, 1, 1], "SAME")
        return np.ascontiguousarray(p.reshape(-1, 9, C).transpose(2, 1, 0))

    Xp, Xqp = patches(act), patches(actq)
    assert np.array_equal(Xp[7], O.channel_patches(act, 7, (3, 3), (2, 2), "SAME"))
    Q = engine.conv_layer_nhwc(act, actq, W, A, **geo)
    Qd = engine.conv_layer_nhwc(torch.from_numpy(act).cuda(), torch.from_numpy(actq).cuda(), torch.from_numpy(W).cuda(), A, **geo)
    assert np.array_equal(Qd.cpu().numpy(), Q)
    assert O.agreement(Q, c_oracle.quantize_conv_layer(W, lambda c: (Xp[c], Xqp[c]), A)) == 1.0
    # the two calls cut the patch columns into different partial slots (two image chunks against one), so their fp64 sums are
    # associated differently and the Grams may differ in the last bits: each is held to the bound against NumPy instead
    gram = engine.conv_gram_nhwc(act, actq, (3, 3), **geo)
    gram_d = engine.conv_gram_nhwc(torch.from_numpy(act).cuda(), torch.from_numpy(actq).cuda(), (3, 3), **geo)
    _assert_grams(gram, list(zip(Xp, Xqp)))
    _assert_grams(gram_d, list(zip(Xp, Xqp)))
    assert np.array_equal(engine.conv_layer_from_gram(gram, W, A), Q)
