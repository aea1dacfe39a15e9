"""The reference's OWN host code as the whole-network oracle (SURVEY.md 8f row 2).

`oracle/ref_shim.py` maps the TensorFlow / h5py names `scripts/quantized_network.py` imports onto NumPy stand-ins
(`hostnet` layers / Model / clone_model / extract_patches, an in-memory h5py.File with create_dataset / resize / slicing),
so that the UNMODIFIED reference file runs here:

  * `QuantizedNeuralNetwork(...).quantize_network()` (:576-590) end to end -- `_get_layer_data_generator` (:408-502, with
    its short-final-batch row arithmetic :491-495), `_quantize_layer_parallel` (:523-574), `_update_weights` (:504-521);
  * for conv layers `_get_layer_data_generator`, `_build_patch_array` (:729-809) and `_quantize_channel_parallel_jit`
    (:652-727) called directly (`_quantize_conv2D_layer_parallel_jit` itself raises on NumPy >= 1.25 at :835-837).

Those reference runs are stored as golden files (oracle/make_golden.py -> tests/golden/ref_network_*.npz,
ref_layer_data.npz).  CPU tests: this repo's mirror classes, driven by the oracle engine, must reproduce the reference's
layer data and quantized weights exactly -- a check of the mirror's re-typed host logic against the reference's, not
against itself.  GPU tests: the mirror on the CUDA path against the same golden files.
"""
import os

import numpy as np
import pytest

from conftest import golden
from oracle import c_oracle, gpfq_oracle as O, ref_shim
from quantized_neural_networks_b200 import QuantizedCNN, QuantizedNeuralNetwork, hostnet

QUIET = type("L", (), {"info": staticmethod(lambda m: None)})()


class OracleEngine:
    """The engine's call surface with the hot path routed through the C oracle (CPU)."""
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

    def conv_layer_nhwc(self, act, actq, W, A, strides=(1, 1), padding="SAME", rate=(1, 1), c0=0, n_channels=None):
        actq = act if actq is None else actq
        kh, kw = W.shape[:2]
        rate = tuple(rate) if rate else (1, 1)
        return c_oracle.quantize_conv_layer(W, lambda c: (O.channel_patches(act, c, (kh, kw), tuple(strides), padding, rate),
                                                          O.channel_patches(actq, c, (kh, kw), tuple(strides), padding, rate)), A)


def with_oracle(cls, *args, **kw):
    q = cls(*args, **kw)
    q.__class__ = type("Oracle" + cls.__name__, (cls,), {"engine": property(lambda self: OracleEngine())})
    return q


# ---- the seeded cases (shared with oracle/make_golden.py) ----------------------------------------------------------
def mlp_case():
    """MNIST-shaped MLP (train_mnist_mlp.py: Flatten, Dense, BN, Dense, BN, Dense), reduced widths; un-normalised integer
    pixels with dead border features; 50 images in batches of 16: the final batch has 2, so rows 32:34 are overwritten and
    the last 14 columns stay zero (SURVEY.md App. E 2)."""
    rng = np.random.default_rng(41)
    net = hostnet.mnist_mlp(seed=3, widths=(48, 24), n_in=196, n_out=10)
    x = (rng.integers(0, 256, (50, 14, 14)) * (rng.random((50, 14, 14)) < 0.4)).astype(np.float32)
    x[:, :2, :] = 0
    return net, hostnet.ArraySequence(x, rng.integers(0, 10, 50), 16), x


def cnn_case():
    """CIFAR10-CNN-shaped net (train_cifar10_cnn.py), reduced; 40 images in batches of 16 (short final batch)."""
    rng = np.random.default_rng(42)
    net = hostnet.cifar10_cnn(seed=5, size=12, widths=(4, 6), dense=16, n_out=10)
    x = rng.random((40, 12, 12, 3)).astype(np.float32)
    return net, hostnet.ArraySequence(x, rng.integers(0, 10, 40), 16), x


def run_reference_mlp(bits, c):
    ref = ref_shim.load()
    net, seq, x = mlp_case()
    with ref_shim.serial_pool():
        q = ref.QuantizedNeuralNetwork(net, 16, seq, logger=QUIET, bits=bits, alphabet_scalar=c)
        q.quantize_network()
    return net, seq, x, q


def run_reference_cnn_layers(bits, c, patch_mini_batch_size=16):
    """Walks the conv / Dense layers in network order with the reference's own methods; returns {layer_idx: Q}."""
    ref = ref_shim.load()
    net, seq, x = cnn_case()
    out = {}
    with ref_shim.serial_pool():
        q = ref.QuantizedCNN(net, 16, seq, logger=QUIET, bits=bits, alphabet_scalar=c, patch_mini_batch_size=patch_mini_batch_size)
        for idx, layer in enumerate(net.layers):
            kind = layer.__class__.__name__
            if kind == "Dense":
                q._quantize_dense_layer(idx)
                out[idx] = np.array(q.quantized_net.layers[idx].get_weights()[0])
            elif kind == "Conv2D":
                hf = q._get_layer_data_generator(idx)                       # :820
                W = layer.get_weights()[0]
                rad = q.alphabet_scalar * np.median(np.abs(W.flatten()))    # :831-832, evaluated literally
                alphabet = rad * q.alphabet
                Q = np.zeros(W.shape)
                for ch in range(W.shape[-2]):                               # the channel loop of :844-860
                    Q[:, :, ch, :] = q._quantize_channel_parallel_jit(ch, W[:, :, ch, :], hf, layer.strides, layer.padding.upper(),
                                                                       layer.dilation_rate, alphabet, patch_mini_batch_size)
                q._update_weights(idx, Q)                                   # :864
                os.remove(f"./{hf}")                                        # :867
                out[idx] = np.array(q.quantized_net.layers[idx].get_weights()[0])
    return net, seq, x, q, out


def reference_quantized_net(net, Q):
    """The quantized network the reference holds after quantizing layers {idx: Q}: a clone carrying the trained weights
    (:377-380) with each quantized layer's kernel replaced and its bias kept (`_update_weights` :504-521)."""
    qnet = hostnet.clone_model(net)
    qnet.set_weights(net.get_weights())
    for idx, Qi in Q.items():
        qnet.layers[idx].set_weights([Qi] + net.layers[idx].get_weights()[1:])
    return qnet


# ---- CPU: mirror (oracle engine) == reference's own host code (its stored outputs) ------------------------------------
@pytest.mark.parametrize("bits,c", [(np.log2(3), 2), (3, 4)])
def test_reference_mlp_quantize_network_vs_mirror(bits, c, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    z = golden("ref_network_mlp")
    tag = ("ternary" if bits == np.log2(3) else f"bits{bits}") + f"_c{c}"
    net, seq, x = mlp_case()
    qm = with_oracle(QuantizedNeuralNetwork, net, 16, seq, logger=QUIET, bits=bits, alphabet_scalar=c)
    qm.quantize_network()
    Qr = {}
    for idx, layer in enumerate(net.layers):
        if layer.__class__.__name__ == "Dense":
            Qr[idx] = z[f"{tag}_Q{idx}"]
            assert np.array_equal(Qr[idx], qm.quantized_net.layers[idx].get_weights()[0]), idx
            assert not np.array_equal(Qr[idx], layer.get_weights()[0])
    assert len(Qr) == 3
    pred = reference_quantized_net(net, Qr).predict(x)
    assert np.array_equal(pred.argmax(-1), z[f"{tag}_pred"])
    assert np.array_equal(pred, qm.quantized_net.predict(x))
    assert not os.listdir(tmp_path)          # no hand-off files left behind (the reference removes its own, :574)


def test_reference_layer_data_generator_short_final_batch(tmp_path, monkeypatch):
    """`_get_layer_data_generator` of the reference (:464-500; its wX / qX stored by oracle/make_golden.py pin_goldens)
    against the mirror's in-memory version, both layouts."""
    monkeypatch.chdir(tmp_path)
    z = golden("ref_layer_data")
    net, seq, x = mlp_case()
    qm = QuantizedNeuralNetwork(net, 16, seq, logger=QUIET)
    for idx, transpose in ((1, True), (3, True), (3, False), (5, True)):
        key = f"{idx}{'t' if transpose else ''}"
        data = qm._get_layer_data_generator(idx, transpose=transpose)
        assert np.array_equal(z["wX" + key], data.wX) and np.array_equal(z["qX" + key], data.qX)
        m = len(seq) * seq.batch_size
        assert (data.wX.shape[-1] if transpose else data.wX.shape[0]) == m == 64
        tail = data.wX[..., 50:] if transpose else data.wX[50:]
        assert not tail.any()                # rows past the overwritten short batch stay zero-filled


def test_reference_cnn_layers_vs_mirror(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    z = golden("ref_network_cnn")
    net, seq, x = cnn_case()
    Qr = {int(k[1:]): z[k] for k in z.files if k.startswith("Q")}
    pred = reference_quantized_net(net, Qr).predict(x)
    assert np.array_equal(pred.argmax(-1), z["pred"])
    for conv_path in ("nhwc", "patches"):
        qm = with_oracle(QuantizedCNN, net, 16, seq, logger=QUIET, bits=4, alphabet_scalar=4, conv_path=conv_path,
                         patch_mini_batch_size=16)
        qm.quantize_network()
        for idx, Q in Qr.items():
            assert np.array_equal(qm.quantized_net.layers[idx].get_weights()[0], Q), (conv_path, idx)
        assert np.array_equal(pred, qm.quantized_net.predict(x))
    assert len(Qr) == 6                      # four conv + two Dense layers


# ---- GPU: mirror on the CUDA path == golden outputs of the reference's own host code --------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tag,bits,c", [("ternary_c2", np.log2(3), 2), ("bits3_c4", 3, 4)])
def test_gpu_mlp_matches_reference_quantize_network(tag, bits, c):
    z = golden("ref_network_mlp")
    net, seq, x = mlp_case()
    q = QuantizedNeuralNetwork(net, 16, seq, logger=QUIET, bits=bits, alphabet_scalar=c)
    q.quantize_network()
    for idx, layer in enumerate(net.layers):
        if layer.__class__.__name__ == "Dense":
            assert np.array_equal(q.quantized_net.layers[idx].get_weights()[0], z[f"{tag}_Q{idx}"]), idx
    assert np.array_equal(q.quantized_net.predict(x).argmax(-1), z[f"{tag}_pred"])


@pytest.mark.gpu
@pytest.mark.parametrize("conv_path", ["nhwc", "patches"])
def test_gpu_cnn_matches_reference_host_code(conv_path):
    z = golden("ref_network_cnn")
    net, seq, x = cnn_case()
    q = QuantizedCNN(net, 16, seq, logger=QUIET, bits=4, alphabet_scalar=4, conv_path=conv_path, patch_mini_batch_size=16)
    q.quantize_network()
    n = 0
    for idx, layer in enumerate(net.layers):
        if layer.__class__.__name__ in ("Dense", "Conv2D"):
            assert np.array_equal(q.quantized_net.layers[idx].get_weights()[0], z[f"Q{idx}"]), idx
            n += 1
    assert n == 6
    assert np.array_equal(q.quantized_net.predict(x).argmax(-1), z["pred"])


# ---- GPU: the reference-side binding of INTEGRATION.md section 1, executed verbatim --------------------------------------
@pytest.mark.gpu
def test_integration_md_stub_runs_as_written(tmp_path, monkeypatch):
    """INTEGRATION.md shows the ~40-line ctypes stub a maintainer of the reference would drop into scripts/gpfq_cuda.py.  This
    test extracts that code block from the document, executes it unchanged (h5py -> the in-memory stand-in of ref_shim, the
    bare "libgpfq.so" resolved to the in-tree build) and drives both of its functions on hand-off files written the way the
    reference writes them (`layer{idx}_data.h5` :471-500, `channel{c}_patch_array.h5` :756-797)."""
    import ctypes
    import re
    import sys
    import types
    from quantized_neural_networks_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "INTEGRATION.md")).read()
    code = re.search(r"## 1\. The stub.*?```python\n(.*?)```", text, re.S).group(1)
    monkeypatch.chdir(tmp_path)
    monkeypatch.setitem(sys.modules, "h5py", types.SimpleNamespace(File=ref_shim._MemFile))
    real_cdll = ctypes.CDLL
    monkeypatch.setattr(ctypes, "CDLL", lambda name, *a, **k: real_cdll(_lib.LIB_PATH if name == "libgpfq.so" else name, *a, **k))
    stub = {}
    exec(compile(code, "INTEGRATION.md#stub", "exec"), stub)

    rng = np.random.default_rng(77)
    N0, N1, m = 300, 12, 640
    Z = rng.standard_normal((N0, m))
    wX = np.maximum(Z, 0).astype(np.float32)
    qX = np.maximum(Z + 0.05 * rng.standard_normal((N0, m)), 0).astype(np.float32)
    W = (rng.uniform(-1, 1, (N0, N1)) * 0.2).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(np.log2(3)))
    with ref_shim._MemFile("layer3_data.h5", "w") as hf:
        hf.create_dataset("wX", shape=(N0, m))
        hf.create_dataset("qX", shape=(N0, m))
        hf["wX"][...] = wX
        hf["qX"][...] = qX
    assert np.array_equal(stub["dense_layer"](W, "layer3_data.h5", A), c_oracle.quantize_layer(W, wX, qX, A))

    act = np.maximum(rng.standard_normal((6, 10, 10, 3)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    Wc = (rng.uniform(-1, 1, (3, 3, 3, 5)) * 0.3).astype(np.float32)
    Ac = O.layer_alphabet(Wc, 4, O.unit_alphabet(4))
    files, pm = [], []
    for c in range(3):
        Xp = O.channel_patches(act, c, (3, 3), (1, 1), "SAME")
        Xqp = O.channel_patches(actq, c, (3, 3), (1, 1), "SAME")
        pm.append((Xp, Xqp))
        with ref_shim._MemFile(f"channel{c}_patch_array.h5", "w") as hf:
            hf.create_dataset(f"wX_channel{c}", data=Xp, chunks=True, maxshape=(None, None))
            hf.create_dataset(f"qX_channel{c}", data=Xqp, chunks=True, maxshape=(None, None))
        files.append(f"channel{c}_patch_array.h5")
    assert np.array_equal(stub["conv_channels"](Wc, files, Ac), c_oracle.quantize_conv_layer(Wc, lambda c: pm[c], Ac))
