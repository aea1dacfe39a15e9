"""GPU: parity of the CUDA path (through the C ABI) with the reference's outputs.

Bars (BASELINE.json north_star): quantized weights identical on >= 99.99 % of entries, mismatches only at
alphabet-boundary ties; per-layer relative residual within 1e-6 (relative) of the oracle's.  On the golden
vectors and small seeded cases we demand EXACT equality: the streaming kernel follows the reference's dtype
ladder operation by operation, and the Gram form only differs at the 1e-9 level of the decision argument.
"""
import numpy as np
import pytest

from conftest import glorot, golden, hidden_pair
from oracle import c_oracle, gpfq_oracle as O

pytestmark = pytest.mark.gpu
AGREE = 0.9999          # north_star: >= 99.99 % of entries
RESID_RTOL = 1e-6       # north_star: relative residual within 1e-6 relative


def check(Q, Qref, W=None, X=None, Xq=None, exact=False):
    agree = O.agreement(Q, Qref)
    if exact:
        assert agree == 1.0, f"agreement {agree}"
    assert agree >= AGREE, f"agreement {agree}"
    if W is not None:
        r, rref = O.relative_residual(W, Q, X, Xq), O.relative_residual(W, Qref, X, Xq)
        assert abs(r - rref) <= RESID_RTOL * max(rref, 1e-30), (r, rref)


# ---- golden vectors (outputs of the unmodified reference) ------------------------------------------
@pytest.mark.parametrize("method", ["stream", "stream_fast", "gram", "auto"])
def test_kat_reference_fixture(engine, method):
    z = golden("kat_settings_fixture")
    X0 = np.ascontiguousarray(z["data"].T)
    for tag in ("t1", "t2", "t3", "b2c2", "b2c3", "b3c2", "b4c5"):
        Q0 = engine.dense_layer(X0, None, z["W0"], z[f"{tag}_A0"], method=method)
        assert np.array_equal(Q0, z[f"{tag}_Q0"]), (tag, Q0)
        Q1 = engine.dense_layer(z[f"{tag}_X1"], z[f"{tag}_Xq1"], z["W1"], z[f"{tag}_A1"], method=method)
        assert np.array_equal(Q1, z[f"{tag}_Q1"]), (tag, Q1)


@pytest.mark.parametrize("method", ["stream", "stream_fast", "gram"])
@pytest.mark.parametrize("name,xq,tags", [("dense_first_ternary", None, ["c1", "c2", "c3", "c6"]),
                                          ("dense_hidden_grid", "Xq", ["k3", "k4", "k8", "k16"]),
                                          ("dense_int_pixels", None, [""]), ("dense_wide_short", "Xq", [""])])
def test_golden_dense(engine, method, name, xq, tags):
    z = golden(name)
    X = z["X"]
    Xq = z[xq] if xq else None
    for tag in tags:
        A = z["A_" + tag] if tag else z["A"]
        Qref = z["Q_" + tag] if tag else z["Q"]
        Q = engine.dense_layer(X, Xq, z["W"], A, method=method)
        check(Q, Qref, z["W"], X, X if Xq is None else Xq, exact=True)
        assert np.all(np.isin(Q, np.concatenate([A, [0.0]])))


@pytest.mark.parametrize("outer", [1, 2])
@pytest.mark.parametrize("name,xq,tags", [("dense_first_ternary", None, ["c1", "c2", "c3", "c6"]),
                                          ("dense_hidden_grid", "Xq", ["k3", "k4", "k8", "k16"]),
                                          ("dense_int_pixels", None, [""]), ("dense_wide_short", "Xq", [""]), ("ties_and_dead", None, ["3", "4"])])
def test_golden_dense_tensor_core_walk(engine, name, xq, tags, outer):
    """The reference's own outputs through the tensor-core range walk (`sweep_walk = 1`; by default it only takes layers of 2048
    directions and more): Gram-row form (`sweep_outer = 1`) and carried residuals (`sweep_outer = 2`, more than 64 directions),
    3 / 4 / 8 / 16 levels, exact ties (integer pixels, the 4 x 4 tie fixture), dead directions -- the flagged steps replay with the
    literal arithmetic, so every entry must match."""
    z = golden(name)
    X = z["X"]
    Xq = z[xq] if xq else None
    engine.set_option("sweep_walk", 1)
    engine.set_option("sweep_outer", outer)
    try:
        for tag in tags:
            A = z["A" + tag] if name == "ties_and_dead" else (z["A_" + tag] if tag else z["A"])
            Qref = z["Q" + tag] if name == "ties_and_dead" else (z["Q_" + tag] if tag else z["Q"])
            Q = engine.dense_layer(X, Xq, z["W"], A, method="gram")
            check(Q, Qref, z["W"], X, X if Xq is None else Xq, exact=True)
    finally:
        engine.set_option("sweep_walk", 0)
        engine.set_option("sweep_outer", 0)


def test_golden_multi_alphabet_batch(engine):
    """Several (bits, c) grid points over the same X, Xq, W in ONE call (config 5)."""
    z = golden("dense_hidden_grid")
    tags = ["k3", "k4", "k8", "k16"]
    for method in ("gram", "stream"):
        Q = engine.dense_layer(z["X"], z["Xq"], z["W"], [z["A_" + t] for t in tags], method=method)
        for a, t in enumerate(tags):
            assert np.array_equal(Q[a], z["Q_" + t]), (method, t)


def test_golden_ties_and_dead(engine):
    z = golden("ties_and_dead")
    for method in ("stream", "gram"):
        assert np.array_equal(engine.dense_layer(z["X"], None, z["W"], z["A3"], method=method), z["Q3"])
        assert np.array_equal(engine.dense_layer(z["X"], None, z["W"], z["A4"], method=method), z["Q4"])


def test_golden_conv_patches(engine):
    z = golden("conv3x3_small")
    Xp, Xqp = list(z["Xp"]), list(z["Xqp"])
    for tag in ("k16", "k3", "k4"):
        Q = engine.conv_channels(Xp, Xqp, z["W"], z["A_" + tag])
        assert np.array_equal(Q, z["Q_" + tag]), tag
    assert np.array_equal(engine.conv_channels(Xp, None, z["W"], z["A_first"]), z["Q_first"])
    Q = engine.conv_channels(Xp, Xqp, z["W"], [z["A_k16"], z["A_k3"], z["A_k4"]])
    for a, tag in enumerate(("k16", "k3", "k4")):
        assert np.array_equal(Q[a], z["Q_" + tag])


def test_golden_conv_nhwc(engine):
    """On-device patch extraction (extract_patches semantics) + channel walk."""
    z = golden("conv3x3_small")
    for tag in ("k16", "k3", "k4"):
        Q = engine.conv_layer_nhwc(z["act"], z["actq"], z["W"], z["A_" + tag], strides=(1, 1), padding="SAME")
        assert np.array_equal(Q, z["Q_" + tag]), tag
    assert np.array_equal(engine.conv_layer_nhwc(z["act"], None, z["W"], z["A_first"]), z["Q_first"])


def test_conv_channel_shards_compose(engine):
    z = golden("conv3x3_small")
    Xp, Xqp = list(z["Xp"]), list(z["Xqp"])
    full = z["Q_k16"]
    a = engine.conv_channels(Xp[:1], Xqp[:1], z["W"], z["A_k16"], c0=0, n_channels=1)
    b = engine.conv_channels(Xp[1:], Xqp[1:], z["W"], z["A_k16"], c0=1, n_channels=2)
    assert np.array_equal(a + b, full)
    c = engine.conv_layer_nhwc(z["act"], z["actq"], z["W"], z["A_k16"], c0=2, n_channels=1)
    assert np.array_equal(c[:, :, 2, :], full[:, :, 2, :]) and np.all(c[:, :, :2, :] == 0)


# ---- Gram stage against fp64 NumPy ----------------------------------------------------------------
@pytest.mark.parametrize("N0,m", [(96, 400), (200, 3001), (784, 5000), (130, 70)])
def test_gram_stage_fp64(engine, N0, m):
    rng = np.random.default_rng(N0 + m)
    X, Xq = hidden_pair(rng, N0, m)
    engine.set_option("gram_kernel", 1)   # the fp64 DMMA contraction (the tcgen05 kernel has its own tests below)
    try:
        G1, G2 = engine.gram_matrices(X, Xq)
        _, G2s = engine.gram_matrices(X, None)
    finally:
        engine.set_option("gram_kernel", 0)
    R1, R2 = O.gram_matrices(X, Xq)
    tri = np.tril_indices(N0)
    for G, R in ((G1, R1), (G2, R2)):
        err = np.max(np.abs(G[tri] - R[tri]) / np.maximum(np.abs(R[tri]), 1e-300))
        assert err < 1e-12, err
    assert np.max(np.abs(G2s[tri] - (X.astype(np.float64) @ X.astype(np.float64).T)[tri])) < 1e-9 * np.max(R2)


# ---- seeded layers vs the C oracle (literal walk) ----------------------------------------------------
SHAPES = [  # (N0, N1, m, bits, c, first-layer?)
    (300, 10, 2500, np.log2(3), 2, False),      # MNIST output layer shape, fewer samples
    (500, 64, 2500, np.log2(3), 3, False),      # MNIST hidden
    (784, 50, 2000, np.log2(3), 2, True),       # MNIST first layer: X == Xq, dead border pixels
    (2048, 16, 1008, 4, 4, False),              # CIFAR dense 2048 -> 128 (a neuron subset), 4-bit
    (128, 10, 5008, 4, 5, False),               # CIFAR output layer, full m
    (1000, 8, 96, np.log2(3), 2, False),        # m << N0 (VGG fc regime)
    (33, 7, 1234, 3, 3, False),                 # ragged everything
    (1, 3, 17, 2, 2, False), (5, 1, 1, np.log2(3), 1, True),
]


@pytest.mark.parametrize("method", ["stream", "stream_fast", "gram"])
@pytest.mark.parametrize("N0,N1,m,bits,c,first", SHAPES)
def test_dense_vs_oracle(engine, method, N0, N1, m, bits, c, first):
    rng = np.random.default_rng(N0 * 7 + N1 * 3 + m)
    if first:
        X = (rng.uniform(0, 1, (N0, m)) * (rng.uniform(0, 1, (N0, m)) < 0.5)).astype(np.float32)
        X[:: max(N0 // 9, 1)] = 0.0
        Xq = X
    else:
        X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    A = O.layer_alphabet(W, c, O.unit_alphabet(bits))
    Qref = c_oracle.quantize_layer(W, X, Xq, A)
    Q = engine.dense_layer(X, None if first else Xq, W, A, method=method)
    check(Q, Qref, W, X, Xq, exact=(method == "stream"))
    assert engine.last_stats["method"] == {"stream": 1, "gram": 2, "stream_fast": 3}[method]
    assert engine.last_stats["kernel_launches"] > 0


def test_dense_neuron_shards_are_bit_identical(engine):
    """Neurons are independent: any split over shards (GPUs) must give the same bits (SURVEY.md 8e)."""
    rng = np.random.default_rng(99)
    X, Xq = hidden_pair(rng, 256, 1500)
    W = glorot(rng, 256, 37)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(np.log2(3)))
    for method in ("stream", "stream_fast", "gram"):
        full = engine.dense_layer(X, Xq, W, A, method=method)
        for world in (2, 4, 8):
            acc = np.zeros_like(full)
            for r in range(world):
                lo, hi = (r * 37) // world, ((r + 1) * 37) // world
                part = engine.dense_layer(X, Xq, W, A, j0=lo, j1=hi, method=method)
                assert np.all(part[:, :lo] == 0) and np.all(part[:, hi:] == 0)
                acc += part
            assert np.array_equal(acc, full), (method, world)


def test_device_pointer_path_matches_host_path(engine):
    import torch
    rng = np.random.default_rng(3)
    X, Xq = hidden_pair(rng, 200, 900)
    W = glorot(rng, 200, 20)
    A = O.layer_alphabet(W, 2, O.unit_alphabet(4))
    for method in ("stream", "gram"):
        Qh = engine.dense_layer(X, Xq, W, A, method=method)
        Qd = engine.dense_layer(torch.from_numpy(X).cuda(), torch.from_numpy(Xq).cuda(), torch.from_numpy(W).cuda(), A,
                                method=method)
        assert np.array_equal(Qd.cpu().numpy(), Qh)


def test_conv_vs_oracle_larger(engine):
    rng = np.random.default_rng(8)
    n_img, H, Wd, C, F = 20, 16, 16, 6, 12
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    W = (rng.uniform(-1, 1, (3, 3, C, F)) * np.sqrt(6 / (9 * C))).astype(np.float32)
    for bits, c, pad, strides in ((4, 4, "SAME", (1, 1)), (np.log2(3), 2, "VALID", (1, 1)), (2, 3, "SAME", (2, 2))):
        A = O.layer_alphabet(W, c, O.unit_alphabet(bits))
        patches = lambda ch: (O.channel_patches(act, ch, (3, 3), strides, pad), O.channel_patches(actq, ch, (3, 3), strides, pad))
        Qref = c_oracle.quantize_conv_layer(W, patches, A)
        Q = engine.conv_layer_nhwc(act, actq, W, A, strides=strides, padding=pad)
        assert O.agreement(Q, Qref) == 1.0, (bits, pad, strides, O.agreement(Q, Qref))
        Xp = [patches(ch)[0] for ch in range(C)]
        Xqp = [patches(ch)[1] for ch in range(C)]
        assert np.array_equal(engine.conv_channels(Xp, Xqp, W, A), Q)


def test_conv_1x1_and_2x2_and_generic_kernel_sizes(engine):
    rng = np.random.default_rng(12)
    n_img, H, Wd, C, F = 8, 9, 9, 3, 4
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    for k in (1, 2, 5):
        W = (rng.uniform(-1, 1, (k, k, C, F)) * 0.5).astype(np.float32)
        A = O.layer_alphabet(W, 2, O.unit_alphabet(np.log2(3)))
        patches = lambda ch: (O.channel_patches(act, ch, (k, k), (1, 1), "SAME"), O.channel_patches(actq, ch, (k, k), (1, 1), "SAME"))
        Qref = c_oracle.quantize_conv_layer(W, patches, A)
        Xp = [patches(ch)[0] for ch in range(C)]
        Xqp = [patches(ch)[1] for ch in range(C)]
        assert np.array_equal(engine.conv_channels(Xp, Xqp, W, A), Qref), k
        # the NHWC entry point takes every kernel size too (5 x 5: device im2col + one Dense problem per channel)
        assert np.array_equal(engine.conv_layer_nhwc(act, actq, W, A), Qref), k
    # 7 x 7 / stride 2 / VALID (the ResNet50 stem geometry) and a channel shard, first layer (X == Xq)
    act = np.maximum(rng.standard_normal((4, 20, 20, 3)), 0).astype(np.float32)
    W = (rng.uniform(-1, 1, (7, 7, 3, 5)) * 0.2).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(2))
    patches = lambda ch: (O.channel_patches(act, ch, (7, 7), (2, 2), "VALID"),) * 2
    Qref = c_oracle.quantize_conv_layer(W, patches, A)
    Q = engine.conv_layer_nhwc(act, None, W, A, strides=(2, 2), padding="VALID", c0=1, n_channels=2)
    assert np.array_equal(Q[:, :, 1:3], Qref[:, :, 1:3]) and not Q[:, :, 0].any()


def test_msq_and_bit_round(engine):
    rng = np.random.default_rng(4)
    W = rng.standard_normal((37, 11)).astype(np.float32)
    for bits in (np.log2(3), 2, 3, 4):
        A = O.layer_alphabet(W, 2, O.unit_alphabet(bits))
        ref = np.array([O.bit_round(w, A) for w in W.flatten()]).reshape(W.shape)
        assert np.array_equal(engine.msq(W, A), ref)
        t = rng.standard_normal(100) * 2
        t[:4] = [(A[0] + A[1]) / 2, (A[-1] + A[-2]) / 2, 100.0, -100.0]  # exact midpoints: ties to the lower index
        assert np.array_equal(engine.bit_round(t, A), np.array([O.bit_round(v, A) for v in t]))


def test_errors_are_reported_not_swallowed(engine):
    from quantized_neural_networks_b200 import GpfqError
    X = np.zeros((4, 8), np.float32)
    W = np.zeros((4, 2), np.float32)
    with pytest.raises(GpfqError):
        engine.dense_layer(X, None, W, np.linspace(-1, 1, 100))  # K > GPFQ_MAX_K
    with pytest.raises(ValueError):
        engine.dense_layer(X, None, np.zeros((5, 2), np.float32), np.array([-1.0, 0, 1]))


def test_full_size_properties_mnist_layer(engine):
    """BASELINE config 1, first layer at full size (784, 500, 25000): properties that need no oracle pass --
    outputs in the alphabet, shard invariance, stream == gram agreement >= 99.99 %, plus a literal-oracle
    check on a seeded neuron subset."""
    rng = np.random.default_rng(1)
    N0, N1, m = 784, 500, 25000
    X = (rng.uniform(0, 1, (N0, m)) * (rng.uniform(0, 1, (N0, m)) < 0.5)).astype(np.float32)
    X[:28] = 0
    W = glorot(rng, N0, N1)
    A = O.layer_alphabet(W, 2, O.unit_alphabet(np.log2(3)))
    Qg = engine.dense_layer(X, None, W, A, method="gram")
    assert np.all(np.isin(Qg, A) | (Qg == 0))
    sub = [0, 17, 123, 499]
    Qs = np.zeros_like(Qg)
    for j in sub:
        Qs += engine.dense_layer(X, None, W, A, j0=j, j1=j + 1, method="stream")
    Wsub = np.ascontiguousarray(W[:, sub])
    Qref = c_oracle.quantize_layer(Wsub, X, X, A)
    assert np.array_equal(Qs[:, sub], Qref)
    assert O.agreement(Qg[:, sub], Qref) >= AGREE


def test_conv_many_patches_both_paths(engine):
    """n_patches beyond one grid sweep of the patch-extraction kernel (> 2048*256 columns): both conv entry
    points against the Gram-form oracle fed with fp64 Grams of torch-unfolded patches."""
    import torch
    rng = np.random.default_rng(21)
    n_img, H, C, F = 640, 32, 2, 8
    act = np.maximum(rng.standard_normal((n_img, H, H, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    W = (rng.uniform(-1, 1, (3, 3, C, F)) * 0.3).astype(np.float32)
    A = O.layer_alphabet(W, 4, O.unit_alphabet(4))
    n = n_img * H * H

    def unfold(a):
        t = torch.from_numpy(a).cuda().permute(3, 0, 1, 2).reshape(C * n_img, 1, H, H)
        p = torch.nn.functional.unfold(t, 3, padding=1)
        return p.reshape(C, n_img, 9, H * H).permute(0, 2, 1, 3).reshape(C, 9, n).contiguous()

    Xp, Xqp = unfold(act), unfold(actq)
    Qref = np.zeros(W.shape)
    for c in range(C):
        xd, qd = Xp[c].double(), Xqp[c].double()
        G1, G2 = (qd @ xd.T).cpu().numpy(), (qd @ qd.T).cpu().numpy()
        Qref[:, :, c, :] = O.gram_quantize_layer(W[:, :, c, :].reshape(9, F), None, None, A, grams=(G1, G2)).reshape(3, 3, F)
    Wd = torch.from_numpy(W).cuda()
    Qp = engine.conv_channels(list(Xp), list(Xqp), Wd, A).cpu().numpy()
    Qn = engine.conv_layer_nhwc(act, actq, W, A)
    assert O.agreement(Qp, Qref) == 1.0, O.agreement(Qp, Qref)
    assert O.agreement(Qn, Qref) == 1.0, O.agreement(Qn, Qref)
    Qn_dev = engine.conv_layer_nhwc(torch.from_numpy(act).cuda(), torch.from_numpy(actq).cuda(), Wd, A).cpu().numpy()
    assert np.array_equal(Qn_dev, Qn)


def test_long_sample_axis_streaming(engine):
    """m beyond the register-resident limit (512 x 16 samples): the shared-memory residual kernel."""
    rng = np.random.default_rng(5)
    N0, N1, m = 40, 6, 9000
    X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(3))
    Qref = c_oracle.quantize_layer(W, X, Xq, A)
    for method in ("stream", "stream_fast"):
        assert np.array_equal(engine.dense_layer(X, Xq, W, A, method=method), Qref)


@pytest.mark.parametrize("J_neurons", [3, 40, 700, 2500])
def test_streaming_neuron_tiles(engine, J_neurons):
    """Every (samples-per-thread, neurons-per-CTA) tile of the register-resident walk: wide layers put up to 8
    neurons in one CTA; the tiling must not change a single bit (neurons are independent)."""
    rng = np.random.default_rng(J_neurons)
    N0 = 24
    for m in (700, 1504, 2600, 3900, 5008, 8000):
        X, Xq = hidden_pair(rng, N0, m)
        W = glorot(rng, N0, J_neurons)
        A = O.layer_alphabet(W, 2, O.unit_alphabet(np.log2(3)))
        Qref = c_oracle.quantize_layer(W, X, Xq, A)
        assert np.array_equal(engine.dense_layer(X, Xq, W, A, method="stream"), Qref), m
        assert O.agreement(engine.dense_layer(X, Xq, W, A, method="stream_fast"), Qref) >= AGREE, m


def test_conv_gram_kernel_variants_agree(engine):
    """The three 3x3 patch-Gram kernels (TMA-staged, direct LDG, generic) produce the same quantized kernel, on
    ragged column counts (tail stages, several chunks) and on the unaligned fallback (n % 4 != 0)."""
    import torch
    rng = np.random.default_rng(77)
    C, F = 3, 5
    W = (rng.uniform(-1, 1, (3, 3, C, F)) * 0.3).astype(np.float32)
    A = O.layer_alphabet(W, 4, O.unit_alphabet(4))
    for n in (4, 516, 70000, 300004, 70001):
        Xp = np.maximum(rng.standard_normal((C, 9, n)), 0).astype(np.float32)
        Xqp = np.maximum(Xp + 0.05 * rng.standard_normal(Xp.shape), 0).astype(np.float32)
        Qref = np.zeros(W.shape)
        for c in range(C):
            G1 = Xqp[c].astype(np.float64) @ Xp[c].astype(np.float64).T
            G2 = Xqp[c].astype(np.float64) @ Xqp[c].astype(np.float64).T
            Qref[:, :, c, :] = O.gram_quantize_layer(W[:, :, c, :].reshape(9, F), None, None, A, grams=(G1, G2)).reshape(3, 3, F)
        outs = {}
        for variant, kernel in (("tma", 0), ("ldg", 1), ("generic", 2)):
            with _conv_options(engine, conv_kernel=kernel):
                outs[variant] = engine.conv_channels(list(Xp), list(Xqp), W, A)
                same = engine.conv_channels(list(Xqp), None, W, A)
                dev = engine.conv_channels([torch.from_numpy(x).cuda() for x in Xp], [torch.from_numpy(x).cuda() for x in Xqp],
                                           torch.from_numpy(W).cuda(), A).cpu().numpy()
                assert np.array_equal(dev, outs[variant]), (variant, n)
                outs[variant + "_same"] = same
        assert O.agreement(outs["tma"], Qref) == 1.0, n
        assert np.array_equal(outs["tma"], outs["ldg"]) and np.array_equal(outs["tma"], outs["generic"]), n
        assert np.array_equal(outs["tma_same"], outs["ldg_same"]) and np.array_equal(outs["tma_same"], outs["generic_same"]), n


@pytest.mark.parametrize("n_img,H,Wd,C,F,pad", [(5, 7, 12, 5, 4, "SAME"), (9, 10, 8, 8, 3, "VALID"), (3, 32, 32, 16, 6, "SAME"),
                                                (70, 6, 6, 3, 2, "VALID"), (2, 40, 44, 12, 2, "SAME"),
                                                (4, 14, 14, 8, 3, "SAME"), (3, 9, 7, 4, 2, "SAME"), (6, 5, 5, 9, 2, "VALID")])
def test_conv_nhwc_fused_matches_patch_path(engine, n_img, H, Wd, C, F, pad):
    """The fused NHWC kernel (planes in shared memory, no patch matrices) against the im2col + patch-Gram path and the
    oracle: ragged channel groups (scalar loader), full groups (LDG.128 loader), SAME / VALID, several bands, output widths that
    are not a multiple of four (VGG block 5 is 14 x 14)."""
    import torch
    rng = np.random.default_rng(n_img * 31 + C)
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    W = (rng.uniform(-1, 1, (3, 3, C, F)) * 0.3).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(3))
    patches = lambda ch: (O.channel_patches(act, ch, (3, 3), (1, 1), pad), O.channel_patches(actq, ch, (3, 3), (1, 1), pad))
    Qref = c_oracle.quantize_conv_layer(W, patches, A)
    outs = {}
    for variant, kernel in (("tma", 0), ("ldg", 1)):
        with _conv_options(engine, conv_kernel=kernel):
            outs[variant] = engine.conv_layer_nhwc(act, actq, W, A, padding=pad)
            outs[variant + "_same"] = engine.conv_layer_nhwc(actq, None, W, A, padding=pad)
            dev = engine.conv_layer_nhwc(torch.from_numpy(act).cuda(), torch.from_numpy(actq).cuda(), torch.from_numpy(W).cuda(),
                                         A, padding=pad).cpu().numpy()
            assert np.array_equal(dev, outs[variant])
            part = engine.conv_layer_nhwc(act, actq, W, A, padding=pad, c0=1, n_channels=C - 2)
            assert np.array_equal(part[:, :, 1:C - 1], outs[variant][:, :, 1:C - 1]) and np.all(part[:, :, 0] == 0)
    assert O.agreement(outs["tma"], Qref) == 1.0
    assert np.array_equal(outs["tma"], outs["ldg"]) and np.array_equal(outs["tma_same"], outs["ldg_same"])


class _conv_options:
    """Planner overrides of the NHWC conv entry point for a block (gpfq_set_option), restored on exit."""

    def __init__(self, engine, **opts):
        self.engine, self.opts = engine, opts

    def __enter__(self):
        for k, v in self.opts.items():
            self.engine.set_option(k, v)

    def __exit__(self, *exc):
        for k in self.opts:
            self.engine.set_option(k, 0)


@pytest.mark.parametrize("n_img,H,Wd,C,F", [(2, 1, 9, 9, 2), (5, 2, 2, 33, 3), (4, 7, 7, 40, 2), (3, 14, 14, 64, 4),
                                            (2, 28, 28, 96, 2), (2, 16, 16, 32, 3), (1, 45, 37, 36, 2), (70, 8, 8, 44, 2),
                                            (3, 6, 5, 32, 2), (2, 9, 23, 72, 2), (5, 10, 6, 40, 3), (2, 5, 12, 32, 2),
                                            (5, 9, 11, 3, 4), (40, 12, 12, 8, 2), (7, 8, 8, 12, 2), (3, 10, 10, 33, 2),
                                            (33, 6, 7, 16, 2), (2, 70, 66, 3, 2), (2, 19, 56, 32, 2), (2, 32, 32, 40, 2), (1, 9, 64, 32, 2)])
def test_conv_corr9_matches_patch_form(engine, n_img, H, Wd, C, F):
    """Correlation form of the 3x3 / stride 1 / SAME Grams (conv_corr.cu: 13 displacement sums per pixel region, added per
    tap) against the oracle and against the patch-form kernel (shared-memory planes), with the planner's choice and with
    both variants forced: TMA boxes straight on the activations, and images packed side by side as virtual channels.
    Degenerate images keep the patch form; ragged bands for every band height, channel counts that are not a multiple of
    32, channel shards that start off a 16-byte boundary, channels that are zero except on one border (dead directions)."""
    import torch
    rng = np.random.default_rng(n_img * 131 + H * 7 + C)
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    if C >= 12:   # signed activations too: Gram entries with cancellation
        act[..., 3] = rng.standard_normal((n_img, H, Wd)).astype(np.float32)
        actq[..., 3] = act[..., 3] + 0.05 * rng.standard_normal((n_img, H, Wd)).astype(np.float32)
    W = (rng.uniform(-1, 1, (3, 3, C, F)) * 0.3).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(3))
    patches = lambda ch: (O.channel_patches(act, ch, (3, 3), (1, 1), "SAME"), O.channel_patches(actq, ch, (3, 3), (1, 1), "SAME"))
    Qref = c_oracle.quantize_conv_layer(W, patches, A)
    # a second input: channels 1 and 2 are zero except on the bottom row / right column, so tap rows / columns that never
    # sit there are dead directions (exact zeros in the Gram) and the guard of quantized_network.py:83-84 must fire
    act2, actq2 = act.copy(), actq.copy()
    act2[:, :-1, :, 1] = 0
    actq2[:, :-1, :, 1] = 0
    act2[:, :, :-1, 2] = 0
    actq2[:, :, :-1, 2] = 0
    geom = H >= 6 and Wd >= 5                    # a TMA box (6 rows x 5 columns) fits in the image
    mappable = C >= 32 and C % 4 == 0            # 32-channel boxes on a 16-byte channel pitch
    runs = {"planner": (dict(), {0, 4, 5}), "planes": (dict(conv_kernel=3), {0})}
    if geom and mappable:
        runs["direct"] = (dict(corr_small=1, corr_pack=2), {4})
        if Wd in (8, 14, 16, 28, 32, 56, 64):   # these widths take the strip kernel by default: the band kernel on the same images
            runs["direct, band kernel"] = (dict(corr_small=1, corr_pack=2, corr_strip=2), {4})
    if geom:
        runs["packed"] = (dict(corr_pack=1), {5})
    out = {}
    for name, (opts, kernels) in runs.items():
        with _conv_options(engine, **opts):
            Q = engine.conv_layer_nhwc(act, actq, W, A)
            assert engine.last_stats["gram_kernel"] in kernels, (name, engine.last_stats["gram_kernel"])
            assert O.agreement(Q, Qref) >= AGREE, name
            Qs = engine.conv_layer_nhwc(actq, None, W, A)
            dev = engine.conv_layer_nhwc(torch.from_numpy(act).cuda(), torch.from_numpy(actq).cuda(), torch.from_numpy(W).cuda(), A)
            assert np.array_equal(dev.cpu().numpy(), Q), name
            if C >= 10:   # a shard that starts at channel 1
                part = engine.conv_layer_nhwc(act, actq, W, A, c0=1, n_channels=C - 2)
                assert O.agreement(part[:, :, 1:C - 1], Q[:, :, 1:C - 1]) >= AGREE and np.all(part[:, :, 0] == 0), name
            Q2 = engine.conv_layer_nhwc(act2, actq2, W, A)
            if H >= 2 and Wd >= 2:
                assert np.all(Q2[0, :, 1, :] == 0) and np.all(Q2[:, 0, 2, :] == 0), name   # dead directions: literal zeros
            out[name] = (Q, Qs, Q2)
    for name in out:
        for x, y in zip(out[name], out["planes"]):
            assert O.agreement(x, y) >= AGREE, name


@pytest.mark.parametrize("n_img,C", [(22, 32), (200, 3)])
def test_conv_corr9_host_image_chunks(engine, n_img, C):
    """Host activations larger than one staging chunk (several image chunks, each with its own slot range; whole groups
    of packed images when C = 3) and a full VGG-like plane size: correlation form == patch form == device-pointer call."""
    import torch
    rng = np.random.default_rng(5)
    H, Wd, F = 224, 224, 2
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C), dtype=np.float32), 0)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape, dtype=np.float32), 0)
    W = (rng.uniform(-1, 1, (3, 3, C, F)) * 0.3).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(np.log2(3)))
    Q = engine.conv_layer_nhwc(act, actq, W, A)
    assert engine.last_stats["gram_kernel"] == (4 if C == 32 else 5)
    dev = engine.conv_layer_nhwc(torch.from_numpy(act).cuda(), torch.from_numpy(actq).cuda(), torch.from_numpy(W).cuda(), A)
    assert np.array_equal(dev.cpu().numpy(), Q) or O.agreement(dev.cpu().numpy(), Q) >= AGREE
    engine.set_option("conv_kernel", 3)
    try:
        Qp = engine.conv_layer_nhwc(act, actq, W, A)
    finally:
        engine.set_option("conv_kernel", 0)
    assert O.agreement(Q, Qp) >= AGREE
    assert np.all(np.isin(Q, np.concatenate([A, [0.0]])))


# ---- Dense Gram stage on tcgen05 (int8 slices, gram_i8.cu) ------------------------------------------------------------
class _gram_kernel:
    """Force the Dense Gram kernel for a block: 1 = fp64 DMMA contraction, 2 = int8 slices on tcgen05."""

    def __init__(self, engine, variant, pairs_d=0):
        self.engine, self.variant, self.pairs_d = engine, variant, pairs_d

    def __enter__(self):
        self.engine.set_option("gram_kernel", self.variant)
        self.engine.set_option("i8_pairs_d", self.pairs_d)

    def __exit__(self, *exc):
        self.engine.set_option("gram_kernel", 0)
        self.engine.set_option("i8_pairs_d", 0)


def _gram_inputs(kind, N0, m):
    rng = np.random.default_rng(N0 * 7 + m)
    if kind == "hidden":
        return hidden_pair(rng, N0, m)
    if kind == "signed":   # no ReLU: products of both signs, Gram entries with heavy cancellation
        X = rng.standard_normal((N0, m)).astype(np.float32)
        return X, (X + 0.05 * rng.standard_normal((N0, m))).astype(np.float32)
    if kind == "wide":     # tiny entries next to a few large ones: the slicing kernel must keep every slice pair
        X = (rng.standard_normal((N0, m)) * 1e-4).astype(np.float32)
        X[:, ::97] = 50.0
        return X, (X * (1 + 1e-3 * rng.standard_normal((N0, m)))).astype(np.float32)
    raise ValueError(kind)


@pytest.mark.parametrize("N0,m,kind", [(96, 400, "hidden"), (256, 1024, "hidden"), (300, 3001, "hidden"), (1000, 129, "signed"),
                                       (520, 2048, "wide"), (2048, 1504, "hidden"), (256, 30000, "hidden"),
                                       (1500, 5008, "signed")])
def test_gram_i8_tcgen05_vs_fp64(engine, N0, m, kind):
    """int8-slice Grams (15+ of 25 slice pairs, exact integer accumulation in TMEM) against fp64 NumPy: the error is
    measured against |Xq| |X|^T, the scale every product is rounded at, and must stay far inside the 1e-9 parity budget
    (SURVEY.md App. C).  Covers ragged tiles, K splits (few tiles), several K chunks (m > 26112) and the wide-row switch."""
    X, Xq = _gram_inputs(kind, N0, m)
    A, B = X.astype(np.float64), Xq.astype(np.float64)
    tri = np.tril_indices(N0)
    with _gram_kernel(engine, 2):
        G1, G2 = engine.gram_matrices(X, Xq)
    for G, R, S in ((G2, B @ B.T, np.abs(B) @ np.abs(B).T), (G1, B @ A.T, np.abs(B) @ np.abs(A).T)):
        err = np.max(np.abs(G[tri] - R[tri]) / np.maximum(S[tri], 1e-300))
        assert err < 1e-10, (kind, err)
    with _gram_kernel(engine, 2, pairs_d=10):   # every slice pair: only the 2^-38 slice rounding is left
        _, G2x = engine.gram_matrices(X, Xq)
    assert np.max(np.abs(G2x[tri] - (B @ B.T)[tri]) / np.maximum((np.abs(B) @ np.abs(B).T)[tri], 1e-300)) < 2e-11


def test_gram_i8_is_exact_on_integer_pixels(engine):
    """MNIST-style un-normalised pixels (integers 0..255, dead rows; train_mnist_mlp.py:48-53): the slices hold the values
    exactly and the integer accumulation makes the Gram bit-exact."""
    rng = np.random.default_rng(5)
    N0, m = 784, 6000
    X = (rng.integers(0, 256, (N0, m)) * (rng.random((N0, m)) < 0.4)).astype(np.float32)
    X[:30] = 0
    with _gram_kernel(engine, 2):
        _, G2 = engine.gram_matrices(X, None)
    R = X.astype(np.float64) @ X.astype(np.float64).T
    tri = np.tril_indices(N0)
    assert np.array_equal(G2[tri], R[tri])


@pytest.mark.parametrize("variant", [1, 2])
def test_dense_gram_kernels_match_the_oracle(engine, variant):
    """Gram + sweep with the Gram stage forced onto the DMMA contraction (1) and onto tcgen05 (2): golden vectors exact,
    seeded layers against the literal C oracle, and both kernels give the same quantized layer."""
    with _gram_kernel(engine, variant):
        for name in ("dense_first_ternary", "dense_hidden_grid", "dense_wide_short"):
            z = golden(name)
            Xq = z["Xq"] if "Xq" in z.files else None
            for qk in [k for k in z.files if k == "Q" or k.startswith("Q_")]:
                Q = engine.dense_layer(z["X"], Xq, z["W"], z["A" + qk[1:]], method="gram")
                assert np.array_equal(Q, z[qk]), (name, qk)
        rng = np.random.default_rng(321)
        for N0, N1, m, first in ((784, 40, 3000, True), (512, 24, 2500, False), (2048, 12, 1504, False)):
            if first:
                X = (rng.uniform(0, 1, (N0, m)) * (rng.uniform(0, 1, (N0, m)) < 0.5)).astype(np.float32)
                X[:20] = 0
                Xq = X
            else:
                X, Xq = hidden_pair(rng, N0, m)
            W = glorot(rng, N0, N1)
            A = O.layer_alphabet(W, 3, O.unit_alphabet(4))
            Qref = c_oracle.quantize_layer(W, X, Xq, A)
            Q = engine.dense_layer(X, None if first else Xq, W, A, method="gram")
            assert engine.last_stats["gram_kernel"] == variant
            check(Q, Qref, W, X, Xq, exact=True)


# ---- sweep with carried residuals (low-rank outer level, m << N0: VGG16 fc1 regime) ------------------------------------
@pytest.mark.parametrize("N0,N1,m,first", [(1000, 8, 96, False), (2304, 40, 200, False), (1500, 300, 64, True), (700, 20, 1500, False),
                                           (600, 2200, 64, False), (520, 2048, 48, True)])
def test_sweep_lowrank_outer_level_matches_the_oracle(engine, N0, N1, m, first):
    """`sweep_outer = 2`: the earlier ranges enter through the residuals U (nj x m) instead of Gram rows, and only
    block-diagonal Gram tiles exist.  Same decisions as the literal oracle walk and as the Gram-row form; the int8 form
    (tensor-core walk) and the fp64 form (sweep_pipe / sweep_tile) agree bit for bit on every alphabet."""
    rng = np.random.default_rng(N0 + N1 + m)
    if first:
        X = (rng.uniform(0, 1, (N0, m)) * (rng.uniform(0, 1, (N0, m)) < 0.5)).astype(np.float32)
        X[:10] = 0
        Xq = X
    else:
        X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    A = O.layer_alphabet(W, 2, O.unit_alphabet(np.log2(3)))
    Qref = c_oracle.quantize_layer(W, X, Xq, A)
    engine.set_option("sweep_outer", 2)
    try:
        Q = engine.dense_layer(X, None if first else Xq, W, A, method="gram")       # contractions on tcgen05 (int8 slices)
        assert engine.last_stats["gram_kernel"] == 3 and (engine.last_stats["reserved"] & 3) == 3   # ... and sweep_tc_kernel
        A2 = O.layer_alphabet(W, 4, O.unit_alphabet(3))
        Qm = engine.dense_layer(X, None if first else Xq, W, [A, A2], method="gram", j0=1, j1=N1 - 1)
        # alphabets with more than three levels through the tensor-core walk (even K: no zero level; the 16 levels of 4 bits)
        Q16 = {bits: engine.dense_layer(X, None if first else Xq, W, O.layer_alphabet(W, 3, O.unit_alphabet(bits)), method="gram")
               for bits in (2, 4)}
        engine.set_option("sweep_i8", 2)                                            # the same on the fp64 DMMA pipe, the ranges
        try:                                                                        # walked by sweep_pipe / sweep_tile
            Qf = engine.dense_layer(X, None if first else Xq, W, A, method="gram")
            assert engine.last_stats["gram_kernel"] == 3 and not engine.last_stats["reserved"] & 3
            for bits, Qb in Q16.items():
                Ab = O.layer_alphabet(W, 3, O.unit_alphabet(bits))
                assert np.array_equal(engine.dense_layer(X, None if first else Xq, W, Ab, method="gram"), Qb)
        finally:
            engine.set_option("sweep_i8", 0)
        assert np.array_equal(Q, Qf)
    finally:
        engine.set_option("sweep_outer", 0)
    for bits, Qb in Q16.items():
        # (520, 2048, m = 48) with 16 levels: ONE neuron meets a tie at the 1e-9 level of the Gram form and leaves the oracle's path
        # there (132 of 1 064 960 entries) -- every walk kernel alike
        Ab = O.layer_alphabet(W, 3, O.unit_alphabet(bits))
        assert O.agreement(Qb, c_oracle.quantize_layer(W, X, Xq, Ab)) >= 0.9998
    check(Q, Qref, W, X, Xq, exact=True)
    engine.set_option("sweep_outer", 1)
    try:
        Qg = engine.dense_layer(X, None if first else Xq, W, A, method="gram")
    finally:
        engine.set_option("sweep_outer", 0)
    assert np.array_equal(Q, Qg)
    assert np.array_equal(Qm[0][:, 1:N1 - 1], Q[:, 1:N1 - 1])      # batched alphabets + a neuron shard
    if N1 >= 2048:   # the default ran two halves of the neurons on two streams: same bits as one chain
        engine.set_option("sweep_outer", 3)
        try:
            assert np.array_equal(engine.dense_layer(X, None if first else Xq, W, A, method="gram"), Q)
        finally:
            engine.set_option("sweep_outer", 0)
    assert np.array_equal(Qm[1][:, 1:N1 - 1], c_oracle.quantize_layer(W, X, Xq, A2)[:, 1:N1 - 1])


# ---- the tensor-core range walk under the Gram-row form of the sweep (sweep_tc.cu; default from 2048 directions) -----------
@pytest.mark.parametrize("N0,N1,m,first,bits", [(1100, 130, 1500, False, np.log2(3)), (700, 40, 2000, True, 4), (2304, 200, 2600, False, 4),
                                                 (1030, 257, 1200, False, 2)])
def test_tensor_core_walk_gram_rows(engine, N0, N1, m, first, bits):
    """`sweep_walk = 1` with `sweep_outer = 1`: what the earlier ranges contribute comes from the Gram-row contraction, the range itself
    is walked by sweep_tc_kernel (ragged last range, neuron counts off the 128 grid, dead directions, 3 / 4 / 16 levels).  Same layer as
    the oracle's literal walk and as sweep_pipe / sweep_tile."""
    rng = np.random.default_rng(N0 + N1 + m)
    if first:
        X = (rng.uniform(0, 1, (N0, m)) * (rng.uniform(0, 1, (N0, m)) < 0.5)).astype(np.float32)
        X[5:25] = 0
        Xq = X
    else:
        X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    W[:, 5] = 0          # a pruned neuron: its residual stays 0, the :86 guard fires at every step (every block of its warp replays)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(bits))
    engine.set_option("sweep_outer", 1)
    try:
        engine.set_option("sweep_walk", 1)
        Q = engine.dense_layer(X, None if first else Xq, W, A, method="gram")
        Qs = engine.dense_layer(X, None if first else Xq, W, A, method="gram", j0=3, j1=N1 - 2)
        engine.set_option("sweep_walk", 2)
        Qo = engine.dense_layer(X, None if first else Xq, W, A, method="gram")
    finally:
        engine.set_option("sweep_walk", 0)
        engine.set_option("sweep_outer", 0)
    assert np.array_equal(Q, Qo)
    assert np.array_equal(Qs[:, 3:N1 - 2], Q[:, 3:N1 - 2])
    check(Q, c_oracle.quantize_layer(W, X, Xq, A), W, X, Xq, exact=True)


# ---- the int8-slice tcgen05 contraction of the residual-form sweep (slgemm_i8.cu) ---------------------------------------
@pytest.mark.parametrize("M,N,K,tb", [(128, 128, 128, False), (200, 300, 1000, False), (130, 260, 5000, True), (64, 70, 30000, False),
                                      (257, 129, 384, True), (1, 1, 1, False)])
def test_slgemm_i8_matches_fp64(engine, M, N, K, tb):
    """C = A B^T, A fp64 (residual-like: wide dynamic range inside a row), B fp32: D = 7 keeps the dropped slice pairs below
    2^-46 of 2^(eA + eB) per K position; D = 10 (every pair) leaves only the 2^-38 slice rounding; integer data is exact."""
    rng = np.random.default_rng(M * N + K)
    A = rng.standard_normal((M, K)) * np.exp(rng.uniform(-3, 3, (M, K)))
    B = np.maximum(rng.standard_normal((N, K)), 0).astype(np.float32)
    Bin = np.ascontiguousarray(B.T) if tb else B
    ref = A @ B.astype(np.float64).T
    scale = np.abs(A) @ np.abs(B).astype(np.float64).T + 1e-300
    for D, tol in ((6, 5e-9), (7, 5e-11), (10, 5e-11)):
        C = engine.debug_slgemm(A, Bin, D=D, transposed_b=tb)
        err = float(np.max(np.abs(C - ref) / scale))
        assert err <= tol, (D, err)
    Ai = rng.integers(-100, 100, (M, K)).astype(np.float64)
    Bi = rng.integers(0, 255, (N, K)).astype(np.float32)
    Ci = engine.debug_slgemm(Ai, np.ascontiguousarray(Bi.T) if tb else Bi, D=10, transposed_b=tb)
    assert np.array_equal(Ci, Ai @ Bi.astype(np.float64).T)


# ---- streaming vs Gram vs carried residuals: picked by measurement -------------------------------------------------------
def test_auto_picks_a_measured_best_method(engine):
    """BASELINE north_star: the streaming variant "is benchmarked against it per layer shape, and the faster one is picked by
    measurement".  On Dense shapes of configs 1-4 `auto` must stay within 10 % (+ 50 us) of the fastest method measured here
    (tools/dense_methods.py; the full table is profiles/dense_methods_r2.md), and every method must give the same layer."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import dense_methods as DM
    for shape in DM.SHAPES:
        if shape[1] * shape[2] > 4096 * 4096 or shape[1] > 8192:     # the two largest shapes: table only
            continue
        res = DM.measure(engine, shape, reps=2)
        best = min(v["ms"] for k, v in res.items() if k != "auto")
        assert res["auto"]["ms"] <= 1.10 * best + 0.05, (shape, res)
        assert min(v["agreement"] for v in res.values()) >= AGREE, (shape, res)


def test_gram_i8_non_finite_inputs_give_nan_not_garbage(engine):
    """An Inf / NaN in the layer inputs (a diverged activation collection) must not be sliced into finite digits: the tcgen05
    Gram comes back all-NaN, like the fp64 contraction makes of the affected rows."""
    rng = np.random.default_rng(3)
    X = np.maximum(rng.standard_normal((300, 2048)), 0).astype(np.float32)
    for bad in (np.inf, np.nan):
        Xb = X.copy()
        Xb[17, 100] = bad
        with _gram_kernel(engine, 2):
            G1, G2 = engine.gram_matrices(Xb)
        assert np.isnan(G2[np.tril_indices(G2.shape[0])]).all()
