"""CPU: pin the oracle (NumPy + C restatements) to the reference's outputs.

* against the committed golden vectors (outputs of the UNMODIFIED reference, oracle/make_golden.py)
* against the reference itself when GPFQ_REFERENCE_ROOT points at a checkout of it
"""
import numpy as np
import pytest

from conftest import glorot, golden, hidden_pair
from oracle import c_oracle, gpfq_oracle as O, ref_shim


def test_unit_alphabet_levels():
    # quantized_network.py:396 -- K = round(2**bits): 3, 4, 8, 16; even K has no zero level
    for bits, K in ((np.log2(3), 3), (2, 4), (3, 8), (4, 16)):
        a = O.unit_alphabet(bits)
        assert len(a) == K and a[0] == -1 and a[-1] == 1 and a.dtype == np.float64
        assert np.all(np.diff(a) > 0)
        assert (0.0 in a) == (K % 2 == 1)


def test_bit_round_ties_go_to_lower_index():
    a = np.array([-1.0, 0.0, 1.0])
    assert O.bit_round(0.5, a) == 0.0 and O.bit_round(-0.5, a) == -1.0
    assert O.bit_round(7.0, a) == 1.0 and O.bit_round(-7.0, a) == -1.0


def test_kat_reference_fixture_hand_checked():
    """tests/settings.py fixture of the reference (2->3->2 linear, ones kernels): SURVEY.md section 4."""
    z = golden("kat_settings_fixture")
    assert np.all(z["t1_Q0"] == 1) and np.all(z["t1_Q1"] == 1)
    assert np.all(z["t2_Q0"] == 0) and np.all(z["t2_Q1"] == 0)  # w=1 equidistant from 0 and 2: lower index
    assert np.all(z["t3_Q0"] == 0) and np.all(z["t3_Q1"] == 0)
    assert np.all(z["b2c2_Q0"] == 0.6666666666666665)
    assert z["b2c2_Q1"].tolist() == [[0.6666666666666665] * 2, [2.0, 2.0], [2.0, 2.0]]
    assert np.all(z["b2c3_Q0"] == 0.9999999999999998) and np.all(z["b2c3_Q1"] == 0.9999999999999998)


@pytest.mark.parametrize("impl", ["numpy", "c"])
def test_oracle_reproduces_kat_fixture(impl):
    z = golden("kat_settings_fixture")
    X0 = np.ascontiguousarray(z["data"].T)
    run = (lambda W, X, Xq, A: O.quantize_dense_layer(W, X, Xq, A)) if impl == "numpy" else \
        (lambda W, X, Xq, A: c_oracle.quantize_layer(W, X, Xq, A))
    for tag in ("t1", "t2", "t3", "b2c2", "b2c3", "b3c2", "b4c5"):
        assert np.array_equal(run(z["W0"], X0, X0, z[f"{tag}_A0"]), z[f"{tag}_Q0"]), tag
        assert np.array_equal(run(z["W1"], z[f"{tag}_X1"], z[f"{tag}_Xq1"], z[f"{tag}_A1"]), z[f"{tag}_Q1"]), tag


DENSE_CASES = [("dense_first_ternary", None, [f"c{c}" for c in (1, 2, 3, 6)]),
               ("dense_hidden_grid", "Xq", ["k3", "k4", "k8", "k16"]),
               ("dense_int_pixels", None, [""]), ("dense_wide_short", "Xq", [""])]


@pytest.mark.parametrize("impl", ["numpy", "c", "gram"])
@pytest.mark.parametrize("name,xq,tags", DENSE_CASES)
def test_oracle_matches_golden_dense(impl, name, xq, tags):
    z = golden(name)
    X = z["X"]
    Xq = z[xq] if xq else X
    for tag in tags:
        A = z["A_" + tag] if tag else z["A"]
        Qref = z["Q_" + tag] if tag else z["Q"]
        if impl == "numpy":
            Q = O.quantize_dense_layer(z["W"], X, Xq, A)
        elif impl == "c":
            Q = c_oracle.quantize_layer(z["W"], X, Xq, A)
        else:
            Q = O.gram_quantize_layer(z["W"], X, Xq, A)
        assert np.array_equal(Q, Qref), f"{name}/{tag}: agreement {O.agreement(Q, Qref)}"


@pytest.mark.parametrize("impl", ["numpy", "c"])
def test_oracle_matches_golden_conv(impl):
    z = golden("conv3x3_small")
    W = z["W"]
    for tag, first in (("k16", False), ("k3", False), ("k4", False), ("first", True)):
        A = z["A_" + tag]
        patches = (lambda c: (z["Xp"][c], z["Xp"][c])) if first else (lambda c: (z["Xp"][c], z["Xqp"][c]))
        Q = O.quantize_conv_layer(W, patches, A) if impl == "numpy" else c_oracle.quantize_conv_layer(W, patches, A)
        assert np.array_equal(Q, z["Q_" + tag]), tag


def test_oracle_ties_and_dead_directions():
    z = golden("ties_and_dead")
    for A, Q in ((z["A3"], z["Q3"]), (z["A4"], z["Q4"])):
        assert np.array_equal(O.quantize_dense_layer(z["W"], z["X"], z["X"], A), Q)
        assert np.array_equal(c_oracle.quantize_layer(z["W"], z["X"], z["X"], A), Q)
    assert np.all(z["Q4"][2] == 0.0)  # dead direction -> literal 0 even though 0 is not a level (App. E 5)


def test_channel_patches_matches_golden_im2col():
    z = golden("conv3x3_small")
    for c in range(3):
        assert np.array_equal(O.channel_patches(z["act"], c, (3, 3), (1, 1), "SAME"), z["Xp"][c])
        assert np.array_equal(O.channel_patches(z["actq"], c, (3, 3), (1, 1), "SAME"), z["Xqp"][c])


def test_c_oracle_equals_numpy_oracle_midsize():
    rng = np.random.default_rng(5)
    X, Xq = hidden_pair(rng, 160, 1200)
    X[3] = 0
    Xq[3] = 0
    W = glorot(rng, 160, 24)
    for bits, c in ((np.log2(3), 2), (4, 4)):
        A = O.layer_alphabet(W, c, O.unit_alphabet(bits))
        Qn = O.quantize_dense_layer(W, X, Xq, A)
        assert np.array_equal(c_oracle.quantize_layer(W, X, Xq, A), Qn)
        assert O.agreement(O.gram_quantize_layer(W, X, Xq, A), Qn) >= 0.9999


def test_neurons_are_independent_of_sharding():
    rng = np.random.default_rng(6)
    X, Xq = hidden_pair(rng, 64, 300)
    W = glorot(rng, 64, 10)
    A = O.layer_alphabet(W, 2, O.unit_alphabet(np.log2(3)))
    full = c_oracle.quantize_layer(W, X, Xq, A)
    parts = c_oracle.quantize_layer(W, X, Xq, A, 0, 4) + c_oracle.quantize_layer(W, X, Xq, A, 4, 10)
    assert np.array_equal(full, parts)


def test_numpy_oracle_bit_identical_to_reference_dense():
    """`_quantize_neuron_parallel` of the reference (its outputs stored by oracle/make_golden.py pin_goldens)."""
    z = golden("ref_neuron_pins")
    X, Xq, W = z["X"], z["Xq"], z["W"]
    for i, (bits, c) in enumerate(((np.log2(3), 1), (np.log2(3), 3), (2, 2), (3, 4), (4, 6))):
        A = O.layer_alphabet(W, c, O.unit_alphabet(bits))
        assert np.array_equal(A, z[f"A{i}"])
        for j in range(W.shape[1]):
            assert np.array_equal(z[f"Q{i}"][:, j], O.quantize_neuron(W[:, j], X, Xq, A)), (i, j)
        assert np.array_equal(A, (c * np.median(np.abs(W.flatten()))) * np.linspace(-1, 1, int(round(2 ** bits))))


def test_numpy_oracle_bit_identical_to_reference_conv_filter():
    """`_quantize_filter2D_parallel_jit` of the reference (its outputs stored by oracle/make_golden.py pin_goldens)."""
    z = golden("ref_filter_pins")
    for f, Aref, Q in zip(z["F"], z["A"], z["Q"]):
        A = O.layer_alphabet(f, 3, O.unit_alphabet(4))
        assert np.array_equal(A, Aref)
        assert np.array_equal(Q, O.quantize_filter(f, z["Xp"], z["Xqp"], A))


# ---- against the reference itself (only where GPFQ_REFERENCE_ROOT names a checkout) -------------------
needs_ref = pytest.mark.skipif(not ref_shim.available(), reason="reference not present (set GPFQ_REFERENCE_ROOT)")


@needs_ref
def test_golden_vectors_are_current(tmp_path, monkeypatch):
    """The committed fixtures equal what the reference produces today."""
    z = golden("dense_hidden_grid")
    for j in (0, 9):
        assert np.array_equal(ref_shim.ref_quantize_neuron(z["W"][:, j], z["X"], z["Xq"], z["A_k16"]), z["Q_k16"][:, j])
    z = golden("ref_neuron_pins")
    for i in range(5):
        for j in range(z["W"].shape[1]):
            assert np.array_equal(ref_shim.ref_quantize_neuron(z["W"][:, j], z["X"], z["Xq"], z[f"A{i}"]), z[f"Q{i}"][:, j])
    z = golden("ref_filter_pins")
    for f, A, Q in zip(z["F"], z["A"], z["Q"]):
        assert np.array_equal(ref_shim.ref_quantize_filter(f, z["Xp"], z["Xqp"], A), Q)
    import test_reference_host as T
    monkeypatch.chdir(tmp_path)
    z = golden("ref_layer_data")
    net, seq, x = T.mlp_case()
    qr = ref_shim.load().QuantizedNeuralNetwork(net, 16, seq, logger=T.QUIET)
    for idx, transpose in ((1, True), (3, True), (3, False), (5, True)):
        hf = ref_shim.MEMORY_FILES[qr._get_layer_data_generator(idx, transpose=transpose)]
        key = f"{idx}{'t' if transpose else ''}"
        assert np.array_equal(np.asarray(hf["wX"]), z["wX" + key]) and np.array_equal(np.asarray(hf["qX"]), z["qX" + key])
