"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the UNMODIFIED reference.

Run with a checkout of the reference (elybrand/quantized_neural_networks):
    GPFQ_REFERENCE_ROOT=<checkout> python oracle/make_golden.py
Every fixture stores the seeded inputs (X, Xq fp32 feature-major; W fp32; alphabet fp64) and the
output of the reference's own `_quantize_neuron_parallel` (scripts/quantized_network.py:91) or
`_quantize_filter2D_parallel_jit` (:185), executed through oracle/ref_shim.py under the
installed NumPy/SciPy.  The fixtures are small (<= a few hundred KB each) and committed, so the
oracle and the CUDA path stay pinned to the reference on machines where it is absent.
"""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def ref_alphabet(W, bits, c):
    # scripts/quantized_network.py:396, :544-545 evaluated literally
    unit = np.linspace(-1, 1, num=int(round(2 ** bits)))
    rad = c * np.median(np.abs(W.flatten()))
    return rad * unit


def ref_dense(W, X, Xq, A):
    Q = np.zeros(W.shape)
    for j in range(W.shape[1]):
        Q[:, j] = ref_shim.ref_quantize_neuron(W[:, j], X, Xq, A)
    return Q


def ref_conv(W, Xp, Xqp, A):
    """W (kh,kw,C,F); Xp/Xqp lists of per-channel (kh*kw, n) patch matrices."""
    Q = np.zeros(W.shape)
    for c in range(W.shape[2]):
        for f in range(W.shape[3]):
            Q[:, :, c, f] = ref_shim.ref_quantize_filter(W[:, :, c, f], Xp[c], Xqp[c], A, channel_idx=c)
    return Q


def save(name, **arrs):
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrs)
    print(f"{name}: " + ", ".join(f"{k}{tuple(np.shape(v))}" for k, v in arrs.items()))


def hidden_pair(rng, N0, m, noise=0.05):
    Z = rng.standard_normal((N0, m))
    X = np.maximum(Z, 0).astype(np.float32)
    Xq = np.maximum(Z + noise * rng.standard_normal((N0, m)), 0).astype(np.float32)
    return X, Xq


def glorot(rng, N0, N1):
    return (rng.uniform(-1, 1, (N0, N1)) * np.sqrt(6.0 / (N0 + N1))).astype(np.float32)


def main():
    if not ref_shim.available():
        sys.exit("reference not present; set GPFQ_REFERENCE_ROOT to a checkout of elybrand/quantized_neural_networks")

    # --- 1. the reference's own fixture (tests/settings.py:25-48): 2 -> 3 -> 2 linear, ones kernels
    data = np.array([[1, 0], [0, 2]], dtype=np.float32)
    W0, W1 = np.ones((2, 3), np.float32), np.ones((3, 2), np.float32)
    kat = {}
    for tag, bits, c in (("t1", np.log2(3), 1), ("t2", np.log2(3), 2), ("t3", np.log2(3), 3),
                         ("b2c2", 2, 2), ("b2c3", 2, 3), ("b3c2", 3, 2), ("b4c5", 4, 5)):
        X0 = np.ascontiguousarray(data.T)
        A0 = ref_alphabet(W0, bits, c)
        Q0 = ref_dense(W0, X0, X0, A0)
        X1 = np.ascontiguousarray((data @ W0).T.astype(np.float32))
        Xq1 = np.ascontiguousarray((data @ Q0.astype(np.float32)).T.astype(np.float32))
        A1 = ref_alphabet(W1, bits, c)
        Q1 = ref_dense(W1, X1, Xq1, A1)
        kat.update({f"{tag}_A0": A0, f"{tag}_Q0": Q0, f"{tag}_X1": X1, f"{tag}_Xq1": Xq1,
                    f"{tag}_A1": A1, f"{tag}_Q1": Q1})
    save("kat_settings_fixture", data=data, W0=W0, W1=W1, **kat)

    # --- 2. first quantized layer: X == Xq, image-like (50% zeros), dead rows, ternary sweep of c
    rng = np.random.default_rng(2020)
    N0, N1, m = 96, 12, 400
    X = (rng.uniform(0, 1, (N0, m)) * (rng.uniform(0, 1, (N0, m)) < 0.5)).astype(np.float32)
    X[[0, 1, 7, 95]] = 0.0  # dead directions (MNIST border pixels)
    W = glorot(rng, N0, N1)
    out = {"X": X, "W": W}
    for c in (1, 2, 3, 6):
        A = ref_alphabet(W, np.log2(3), c)
        out[f"A_c{c}"] = A
        out[f"Q_c{c}"] = ref_dense(W, X, X, A)
    save("dense_first_ternary", **out)

    # --- 3. hidden layer: X != Xq, all four alphabets of the CIFAR grid
    rng = np.random.default_rng(7)
    N0, N1, m = 128, 10, 600
    X, Xq = hidden_pair(rng, N0, m)
    Xq[17] = 0.0  # dead direction in the quantized walk only
    W = glorot(rng, N0, N1)
    out = {"X": X, "Xq": Xq, "W": W}
    for tag, bits, c in (("k3", np.log2(3), 2), ("k4", 2, 3), ("k8", 3, 4), ("k16", 4, 5)):
        A = ref_alphabet(W, bits, c)
        out[f"A_{tag}"] = A
        out[f"Q_{tag}"] = ref_dense(W, X, Xq, A)
    save("dense_hidden_grid", **out)

    # --- 4. un-normalised integer pixels (MNIST scripts feed 0..255), m not a multiple of 4
    rng = np.random.default_rng(11)
    N0, N1, m = 64, 6, 333
    X = (rng.integers(0, 256, (N0, m)) * (rng.uniform(0, 1, (N0, m)) < 0.3)).astype(np.float32)
    X[[0, 63]] = 0.0
    W = glorot(rng, N0, N1)
    A = ref_alphabet(W, np.log2(3), 3)
    save("dense_int_pixels", X=X, W=W, A=A, Q=ref_dense(W, X, X, A))

    # --- 5. wide-and-short (m < N0, the VGG fc regime) and a single neuron
    rng = np.random.default_rng(13)
    N0, N1, m = 300, 3, 40
    X, Xq = hidden_pair(rng, N0, m, noise=0.1)
    W = glorot(rng, N0, N1)
    A = ref_alphabet(W, np.log2(3), 2)
    save("dense_wide_short", X=X, Xq=Xq, W=W, A=A, Q=ref_dense(W, X, Xq, A))

    # --- 6. conv: 3x3, C=3, F=5 over a small NHWC activation, SAME padding, 4-bit and ternary;
    #        patch matrices built by a straightforward im2col (extract_patches semantics, :158-179)
    rng = np.random.default_rng(17)
    n_img, H, Wd, C, F = 6, 8, 8, 3, 5
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)

    def im2col(a, c):
        p = np.zeros((H + 2, Wd + 2), np.float32)
        cols = np.zeros((9, n_img * H * Wd), np.float32)
        for i in range(n_img):
            p[:] = 0
            p[1:-1, 1:-1] = a[i, :, :, c]
            for r in range(3):
                for cc in range(3):
                    cols[r * 3 + cc, i * H * Wd:(i + 1) * H * Wd] = p[r:r + H, cc:cc + Wd].reshape(-1)
        return cols

    Xp = [im2col(act, c) for c in range(C)]
    Xqp = [im2col(actq, c) for c in range(C)]
    Wc = (rng.uniform(-1, 1, (3, 3, C, F)) * np.sqrt(6.0 / (9 * C))).astype(np.float32)
    out = {"act": act, "actq": actq, "W": Wc, "Xp": np.stack(Xp), "Xqp": np.stack(Xqp)}
    for tag, bits, c in (("k16", 4, 4), ("k3", np.log2(3), 2), ("k4", 2, 2)):
        A = ref_alphabet(Wc, bits, c)
        out[f"A_{tag}"] = A
        out[f"Q_{tag}"] = ref_conv(Wc, Xp, Xqp, A)
    # first conv layer: X == Xq
    A = ref_alphabet(Wc, 4, 3)
    out["A_first"] = A
    out["Q_first"] = ref_conv(Wc, Xp, Xp, A)
    save("conv3x3_small", **out)

    # --- 7. exact alphabet-boundary ties and the even-K dead-direction literal 0
    X = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 0, 0], [0, 0, 1, 1]], np.float32)
    W = np.array([[0.5, -0.5, 1.5], [0.25, 0.75, -1.0], [0.3, 0.3, 0.3], [1.0, -0.25, 0.5]], np.float32)
    A3 = np.array([-1.0, 0.0, 1.0])
    A4 = np.array([-1.0, -1 / 3, 1 / 3, 1.0])
    save("ties_and_dead", X=X, W=W, A3=A3, Q3=ref_dense(W, X, X, A3), A4=A4, Q4=ref_dense(W, X, X, A4))


def network_goldens():
    """Whole-network fixtures: the reference's OWN host code (`QuantizedNeuralNetwork(...).quantize_network()` :576-590;
    for conv layers `_get_layer_data_generator` + `_build_patch_array` + `_quantize_channel_parallel_jit`) run unmodified
    over the hostnet stand-ins, on the seeded cases of tests/test_reference_host.py."""
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_reference_host as T
    cwd = os.getcwd()
    os.chdir(tempfile.mkdtemp())
    try:
        out = {}
        for tag, bits, c in (("ternary_c2", np.log2(3), 2), ("bits3_c4", 3, 4)):
            net, seq, x, q = T.run_reference_mlp(bits, c)
            for idx, layer in enumerate(net.layers):
                if layer.__class__.__name__ == "Dense":
                    out[f"{tag}_Q{idx}"] = np.array(q.quantized_net.layers[idx].get_weights()[0])
            out[f"{tag}_pred"] = q.quantized_net.predict(x).argmax(-1)
        save("ref_network_mlp", **out)
        net, seq, x, q, Qr = T.run_reference_cnn_layers(4, 4)
        out = {f"Q{idx}": Q for idx, Q in Qr.items()}
        out["pred"] = q.quantized_net.predict(x).argmax(-1)
        save("ref_network_cnn", **out)
    finally:
        os.chdir(cwd)


PIN_ALPHABETS = ((np.log2(3), 1), (np.log2(3), 3), (2, 2), (3, 4), (4, 6))
LAYER_DATA_CASES = ((1, True), (3, True), (3, False), (5, True))


def pin_goldens():
    """The reference outputs behind the pins of the NumPy oracle (tests/test_oracle.py) and of the mirror's layer data
    (tests/test_reference_host.py):
      ref_neuron_pins  `_quantize_neuron_parallel` (:91) on five neurons over five alphabets, a dead direction in Xq;
      ref_filter_pins  `_quantize_filter2D_parallel_jit` (:185) on four 3x3 channel filters, 4-bit;
      ref_layer_data   the wX / qX `_get_layer_data_generator` (:408-502) writes for the MLP case of
                       tests/test_reference_host.py (50 images in batches of 16: the short final batch), both layouts.
    The committed files were written by this function with the oracle's `quantize_neuron` / `quantize_filter` and the
    mirror's `_get_layer_data_generator` standing in for the reference's: on exactly these seeded inputs the tests compared
    those with the reference itself and found them bit-identical, and none of that code has changed since.  Run with
    GPFQ_REFERENCE_ROOT set, this function rewrites them from the reference, and test_golden_vectors_are_current checks them
    against it."""
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_reference_host as T

    rng = np.random.default_rng(123)
    X, Xq = hidden_pair(rng, 48, 257)
    Xq[11] = 0.0
    W = glorot(rng, 48, 5)
    out = {"X": X, "Xq": Xq, "W": W}
    for i, (bits, c) in enumerate(PIN_ALPHABETS):
        out[f"A{i}"] = ref_alphabet(W, bits, c)
        out[f"Q{i}"] = ref_dense(W, X, Xq, out[f"A{i}"])
    save("ref_neuron_pins", **out)

    rng = np.random.default_rng(321)
    Xp = rng.uniform(0, 1, (9, 777)).astype(np.float32)
    Xqp = (Xp + 0.02 * rng.standard_normal(Xp.shape)).astype(np.float32)
    F = np.stack([rng.uniform(-0.4, 0.4, (3, 3)).astype(np.float32) for _ in range(4)])
    A = np.stack([ref_alphabet(f, 4, 3) for f in F])
    Q = np.stack([ref_shim.ref_quantize_filter(f, Xp, Xqp, a) for f, a in zip(F, A)])
    save("ref_filter_pins", Xp=Xp, Xqp=Xqp, F=F, A=A, Q=Q)

    cwd = os.getcwd()
    os.chdir(tempfile.mkdtemp())       # the reference leaves its hand-off files in the working directory
    try:
        net, seq, x = T.mlp_case()
        qr = ref_shim.load().QuantizedNeuralNetwork(net, 16, seq, logger=T.QUIET)
        out = {}
        for idx, transpose in LAYER_DATA_CASES:
            hf = ref_shim.MEMORY_FILES[qr._get_layer_data_generator(idx, transpose=transpose)]
            key = f"{idx}{'t' if transpose else ''}"
            out["wX" + key], out["qX" + key] = np.asarray(hf["wX"]), np.asarray(hf["qX"])
        save("ref_layer_data", **out)
    finally:
        os.chdir(cwd)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "network":
        network_goldens()
    elif len(sys.argv) > 1 and sys.argv[1] == "pins":
        pin_goldens()
    else:
        main()
        network_goldens()
        pin_goldens()
