"""GPU: the sample-split Gram stage of a multi-GPU job (SURVEY.md 8e item 4, BASELINE.json north_star: "the Gram stage
splits over samples, using an NCCL all-reduce over NVLink").  One-GPU tests sum per-chunk partial Grams by hand (what the
all-reduce does) and sweep from the sum through `gpfq_dense_layer_from_gram`; the two-GPU test runs the real thing under
torchrun / NCCL when the box has two GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import glorot, golden, hidden_pair
from oracle import c_oracle, gpfq_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _split_grams(engine, X, Xq, parts):
    import torch
    m = X.shape[1]
    same = Xq is None
    G1 = G2 = None
    for r in range(parts):
        lo, hi = (r * m) // parts, ((r + 1) * m) // parts
        if hi == lo:
            continue
        if r % 2:   # strided host views of the sample range (what `sample_split_gram` hands over), device outputs
            g1, g2 = engine.gram_matrices(X[:, lo:hi], None if same else Xq[:, lo:hi], device_out=True)
        else:       # device tensors
            xd = torch.from_numpy(np.ascontiguousarray(X[:, lo:hi])).cuda()
            qd = None if same else torch.from_numpy(np.ascontiguousarray(Xq[:, lo:hi])).cuda()
            g1, g2 = engine.gram_matrices(xd, qd)
        assert g1.is_cuda and g2.dtype == torch.float64 and ((g1 is g2) == same)
        G2 = g2.clone() if G2 is None else G2 + g2
        if not same:
            G1 = g1.clone() if G1 is None else G1 + g1
    return (None if same else G1), G2


@pytest.mark.parametrize("parts", [1, 2, 3])
def test_golden_dense_from_split_grams(engine, parts):
    """Golden vectors of the unmodified reference, Gram stage summed over sample chunks: exact equality."""
    for name, xq, tags in [("dense_first_ternary", None, ["c1", "c3"]), ("dense_hidden_grid", "Xq", ["k3", "k4", "k16"]),
                           ("dense_int_pixels", None, [""]), ("ties_and_dead", None, ["3", "4"])]:
        z = golden(name)
        X, Xq = z["X"], (z[xq] if xq else None)
        G1, G2 = _split_grams(engine, X, Xq, parts)
        for tag in tags:
            if name == "ties_and_dead":
                A, Qref = z["A" + tag], z["Q" + tag]
            else:
                A, Qref = (z["A_" + tag], z["Q_" + tag]) if tag else (z["A"], z["Q"])
            Q = engine.dense_layer_from_gram(G1, G2, z["W"], A)
            assert np.array_equal(Q, Qref), (name, tag, parts, O.agreement(Q, Qref))


@pytest.mark.parametrize("N0,N1,m,first,parts", [(300, 64, 4100, False, 2), (784, 40, 6000, True, 4),
                                                 (1100, 24, 9000, False, 8)])
def test_from_split_grams_vs_oracle_and_one_gpu_path(engine, N0, N1, m, first, parts):
    """Seeded layers large enough for the tcgen05 Gram per chunk: >= 99.99 % against the oracle, residual within 1e-6,
    and the same Q as the one-GPU Gram path; neuron shards of the sweep compose bit-identically."""
    import torch
    rng = np.random.default_rng(N0 + parts)
    if first:
        X = (rng.random((N0, m)) * (rng.random((N0, m)) < 0.5)).astype(np.float32)
        Xq = None
    else:
        X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    A = O.layer_alphabet(W, 2, O.unit_alphabet(np.log2(3)))
    G1, G2 = _split_grams(engine, X, Xq, parts)
    Q = engine.dense_layer_from_gram(G1, G2, W, A)
    assert engine.last_stats["gram_kernel"] == 0 and engine.last_stats["method"] == 2
    Qref = c_oracle.quantize_layer(W, X, X if Xq is None else Xq, A)
    assert O.agreement(Q, Qref) >= 0.9999
    r, rref = (O.relative_residual(W, q, X, X if Xq is None else Xq) for q in (Q, Qref))
    assert abs(r - rref) <= 1e-6 * rref
    Q1 = engine.dense_layer(X, Xq, W, A, method="gram")
    assert O.agreement(Q, Q1) >= 0.9999
    # device W / Q, neuron shards, several alphabets in one call
    Wd = torch.from_numpy(W).cuda()
    A2 = O.layer_alphabet(W, 3, O.unit_alphabet(2))
    out = torch.zeros((2, N0, N1), dtype=torch.float64, device="cuda")
    cut = N1 // 3
    engine.dense_layer_from_gram(G1, G2, Wd, [A, A2], j0=0, j1=cut, out=out)
    engine.dense_layer_from_gram(G1, G2, Wd, [A, A2], j0=cut, j1=N1, out=out)
    both = out.cpu().numpy()
    assert np.array_equal(both[0], Q)
    assert np.array_equal(both[1], engine.dense_layer_from_gram(G1, G2, W, A2))


def test_from_gram_argument_errors(engine):
    import torch
    from quantized_neural_networks_b200 import GpfqError
    G = torch.eye(4, dtype=torch.float64, device="cuda")
    W = np.ones((4, 2), np.float32)
    A = np.array([-1.0, 0.0, 1.0])
    with pytest.raises(ValueError):
        engine.dense_layer_from_gram(None, G, np.ones((5, 2), np.float32), A)
    with pytest.raises(TypeError):
        engine.dense_layer_from_gram(None, G.cpu(), W, A)
    with pytest.raises(GpfqError):
        engine.dense_layer_from_gram(None, G, W, A, j0=1, j1=7)
    Q = engine.dense_layer_from_gram(None, G, W, A)       # orthonormal directions: plain rounding of every weight
    assert np.array_equal(Q, np.ones((4, 2)))


def test_two_gpu_nccl_sample_split_job():
    """The real exchange: torchrun, 2 ranks, NCCL.  `tools/multi_gpu_check.py` runs the mirror classes with
    gram_split="samples" and "replicate" and compares both with the unsharded one-GPU pass on every rank."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29731",
                          os.path.join(ROOT, "tools", "multi_gpu_check.py")], capture_output=True, text=True, env=env,
                         timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "MULTI_GPU_CHECK PASS" in res.stdout


@pytest.mark.parametrize("n_img,H,Wd,C,F,pad,parts", [(6, 9, 11, 8, 3, "SAME", 3), (5, 14, 14, 64, 2, "SAME", 2),
                                                      (7, 8, 8, 5, 2, "VALID", 4), (3, 70, 66, 3, 2, "SAME", 2)])
def test_conv_from_image_split_grams(engine, n_img, H, Wd, C, F, pad, parts):
    """Conv layer split over images (what the ranks of a multi-GPU job do): per-channel Grams of image chunks summed by
    hand (= the all-reduce), walks from the sum through gpfq_conv_layer_from_gram -- against the oracle and the one-call
    entry point; every Gram kernel the planner can pick (planes, correlation form, packed, im2col + patch Grams)."""
    import torch
    rng = np.random.default_rng(n_img * 17 + C)
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    W = (rng.uniform(-1, 1, (3, 3, C, F)) * 0.3).astype(np.float32)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(3))
    patches = lambda ch: (O.channel_patches(act, ch, (3, 3), (1, 1), pad), O.channel_patches(actq, ch, (3, 3), (1, 1), pad))
    Qref = c_oracle.quantize_conv_layer(W, patches, A)
    for same in (False, True):
        gram = None
        for r in range(parts):
            lo, hi = (r * n_img) // parts, ((r + 1) * n_img) // parts
            if hi == lo:
                continue
            if r % 2:   # host arrays in, device Grams out
                g = engine.conv_gram_nhwc(actq[lo:hi] if same else act[lo:hi], None if same else actq[lo:hi], (3, 3), padding=pad)
            else:       # device tensors
                a = torch.from_numpy(np.ascontiguousarray(actq[lo:hi] if same else act[lo:hi])).cuda()
                g = engine.conv_gram_nhwc(a, None if same else torch.from_numpy(np.ascontiguousarray(actq[lo:hi])).cuda(), (3, 3),
                                          padding=pad)
            assert g.is_cuda and tuple(g.shape) == (C, 2, 9, 9)
            gram = g.clone() if gram is None else gram + g
        Q = engine.conv_layer_from_gram(gram, W, A)
        Q1 = engine.conv_layer_nhwc(actq if same else act, None if same else actq, W, A, padding=pad)
        assert O.agreement(Q, Q1) >= 0.9999
        if not same:
            assert O.agreement(Q, Qref) >= 0.9999
        # channel shards of the walk and device W / Q
        Wd_ = torch.from_numpy(W).cuda()
        out = torch.zeros((1, 3, 3, C, F), dtype=torch.float64, device="cuda")
        cut = max(1, C // 3)
        engine.conv_layer_from_gram(gram[:cut].contiguous(), Wd_, A, c0=0, n_channels=cut, out=out)
        engine.conv_layer_from_gram(gram[cut:].contiguous(), Wd_, A, c0=cut, n_channels=C - cut, out=out)
        assert np.array_equal(out[0].cpu().numpy(), Q)


def test_golden_conv_from_gram(engine):
    """Golden conv fixture of the unmodified reference through the Gram-only + from-Gram entry points, the Grams summed over
    two image chunks: exact."""
    z = golden("conv3x3_small")
    act, actq, W = z["act"], z["actq"], z["W"]
    half = act.shape[0] // 2
    gram = engine.conv_gram_nhwc(act[:half], actq[:half], (3, 3)) + engine.conv_gram_nhwc(act[half:], actq[half:], (3, 3))
    for tag in ("k16", "k3", "k4"):
        assert np.array_equal(engine.conv_layer_from_gram(gram, W, z["A_" + tag]), z["Q_" + tag]), tag
    g1 = engine.conv_gram_nhwc(act[:half], None, (3, 3)) + engine.conv_gram_nhwc(act[half:], None, (3, 3))
    assert np.array_equal(engine.conv_layer_from_gram(g1, W, z["A_first"]), z["Q_first"])
