"""CPU: host-side logic of the drop-in layer (no compute calls into libgpfq) -- the TF-free Keras stand-in, activation
collection, patch extraction, sharding and the world_size-2 (gloo) gather of Q shards."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import gpfq_oracle as O  # noqa: E402  (tests may use the oracle; the product never does)
from quantized_neural_networks_b200 import hostnet  # noqa: E402
from quantized_neural_networks_b200.quantized_network import (  # noqa: E402
    LayerData, QuantizedCNN, QuantizedNeuralNetwork, shard_range)


def _unfold_patches(act, c, kernel_size, strides, padding, rate):
    """Patch matrix of channel c by torch.nn.functional.unfold on an explicitly padded input, TensorFlow's SAME split
    (pad before = total // 2): a restatement that shares no loop with the oracle or hostnet."""
    import torch
    (kh, kw), (sh, sw), (rh, rw) = kernel_size, strides, rate
    n, H, Wd = act.shape[:3]
    pads = []
    for size, k, s, r in ((Wd, kw, sw, rw), (H, kh, sh, rh)):   # F.pad order: (left, right, top, bottom)
        total = max((-(-size // s) - 1) * s + (k - 1) * r + 1 - size, 0) if padding == "SAME" else 0
        pads += [total // 2, total - total // 2]
    x = torch.nn.functional.pad(torch.from_numpy(np.ascontiguousarray(act[..., c]))[:, None], pads)
    p = torch.nn.functional.unfold(x, (kh, kw), dilation=(rh, rw), stride=(sh, sw))   # (n, kh*kw, Ho*Wo)
    return p.permute(1, 0, 2).reshape(kh * kw, -1).numpy()


@pytest.mark.parametrize("padding,strides,rate", [("SAME", (1, 1), (1, 1)), ("VALID", (1, 1), (1, 1)),
                                                  ("SAME", (2, 2), (1, 1)), ("VALID", (1, 2), (1, 1)),
                                                  ("SAME", (1, 1), (2, 2)), ("SAME", (2, 1), (1, 1)),
                                                  ("VALID", (2, 1), (2, 1)), ("SAME", (1, 3), (1, 2)),
                                                  ("VALID", (1, 3), (2, 3)), ("SAME", (3, 2), (2, 3)),
                                                  ("VALID", (1, 1), (1, 2)), ("SAME", (4, 4), (1, 1))])
def test_extract_patches_matches_oracle_im2col(padding, strides, rate):
    """Three restatements of the patch geometry agree exactly: hostnet.extract_patches, the oracle's loop and torch's unfold,
    for non-square kernels (taps r * kw + col), asymmetric strides and rates, strides beyond the kernel extent, SAME padding
    with a nonzero top / left pad and VALID outputs one pixel high or wide.  The GPU conv tests compare with the oracle."""
    rng = np.random.default_rng(3)
    for shape in ((3, 7, 6, 2), (2, 9, 13, 2)):
        act = rng.standard_normal(shape).astype(np.float32)
        H, Wd = shape[1:3]
        for ks in ((3, 3), (1, 2), (2, 1), (1, 3), (3, 1), (2, 3), (3, 2), (1, 4), (1, 6), (1, 9), (9, 1), (1, 5), (2, 5),
                   (5, 5)):
            if padding == "VALID" and ((ks[0] - 1) * rate[0] + 1 > H or (ks[1] - 1) * rate[1] + 1 > Wd):
                continue
            for c in range(2):
                ch = act[..., c:c + 1]
                p = hostnet.extract_patches(ch, [1, *ks, 1], [1, *strides, 1], [1, *rate, 1], padding)
                mine = p.reshape(-1, p.shape[-1]).T
                ref = O.channel_patches(act, c, ks, strides, padding, rate)
                assert np.array_equal(mine, ref), (shape, ks)
                assert np.array_equal(_unfold_patches(act, c, ks, strides, padding, rate), ref), (shape, ks)


@pytest.mark.parametrize("n,world", [(10, 1), (10, 3), (128, 8), (3, 8), (37, 4)])
def test_shard_range_partitions(n, world):
    seen = []
    for r in range(world):
        lo, hi = shard_range(n, r, world)
        assert 0 <= lo <= hi <= n
        seen += list(range(lo, hi))
    assert seen == list(range(n))
    sizes = [shard_range(n, r, world)[1] - shard_range(n, r, world)[0] for r in range(world)]
    assert max(sizes) - min(sizes) <= 1


def test_constructor_surface_matches_reference():
    """quantized_network.py:332-400 / :594-650: attributes the drivers read, alphabet, cloned twin with equal weights."""
    net = hostnet.mnist_mlp(seed=1, widths=(12, 8), n_in=16, n_out=4)
    x = np.random.default_rng(0).random((6, 4, 4)).astype(np.float32)
    seq = hostnet.ArraySequence(x, np.zeros(6), 3)
    q = QuantizedNeuralNetwork(net, 3, seq, bits=2, alphabet_scalar=3, ignore_layers=[5])
    assert np.array_equal(q.alphabet, np.linspace(-1, 1, 4))
    assert q.alphabet_scalar == 3 and q.bits == 2 and q.ignore_layers == [5]
    assert q.trained_net is net and q.quantized_net is not net
    for a, b in zip(net.get_weights(), q.quantized_net.get_weights()):
        assert np.array_equal(a, b)
    assert set(q.layer_dims) == {1, 3, 5} and q.layer_dims[1] == (16, 12)
    c = QuantizedCNN(hostnet.cifar10_cnn(seed=2, size=8, widths=(2, 3, 4), dense=5, n_out=3), 2,
                     hostnet.ArraySequence(np.zeros((4, 8, 8, 3), np.float32), np.zeros(4), 2))
    assert np.array_equal(c.alphabet, np.array([-1.0, 0.0, 1.0]))
    assert c.patch_mini_batch_size == 5000 and c.is_quantize_conv2d is True


def test_layer_data_collection_dense_and_conv():
    """_get_layer_data_generator (:408-502): wX/qX of the layer's inbound activations, feature-major when transposed."""
    net = hostnet.mnist_mlp(seed=1, widths=(12, 8), n_in=16, n_out=4)
    x = np.random.default_rng(0).random((6, 4, 4)).astype(np.float32)
    q = QuantizedNeuralNetwork(net, 3, hostnet.ArraySequence(x, np.zeros(6), 3))
    d = q._get_layer_data_generator(1, transpose=True)
    assert d.wX.shape == (16, 6) and d.same
    assert np.array_equal(d.wX, x.reshape(6, 16).T)
    # perturb the quantized twin's first Dense layer: layer 3's inputs now differ between the two nets
    W = q.quantized_net.layers[1].get_weights()
    q.quantized_net.layers[1].set_weights([np.round(W[0] * 4) / 4, W[1]])
    d3 = q._get_layer_data_generator(3, transpose=True)
    assert d3.wX.shape == (12, 6) and not d3.same
    assert np.array_equal(d3.wX.T, net.run(x, 0, 2))
    assert np.array_equal(d3.qX.T, q.quantized_net.run(x, 0, 2))

    cnn = hostnet.cifar10_cnn(seed=2, size=8, widths=(2, 3, 4), dense=5, n_out=3)
    xi = np.random.default_rng(1).random((4, 8, 8, 3)).astype(np.float32)
    c = QuantizedCNN(cnn, 2, hostnet.ArraySequence(xi, np.zeros(4), 2))
    dc = c._get_layer_data_generator(2)
    assert dc.wX.shape == (4, 8, 8, 2)
    assert np.array_equal(dc.wX, cnn.run(xi, 0, 1))
    patches = c._build_patch_array(1, (3, 3), (1, 1), "SAME", (1, 1), dc, 3)
    assert np.array_equal(patches["wX_channel1"], O.channel_patches(dc.wX, 1, (3, 3), (1, 1), "SAME"))


def test_layer_alphabet_matches_reference_dtype_ladder():
    """rad = alphabet_scalar * median(|W|) stays float32 for a Python scalar (NEP 50), :544-545."""
    rng = np.random.default_rng(5)
    W = rng.standard_normal((9, 7)).astype(np.float32)
    net = hostnet.mnist_mlp(seed=1, widths=(12, 8), n_in=16, n_out=4)
    q = QuantizedNeuralNetwork(net, 3, hostnet.ArraySequence(np.zeros((2, 4, 4), np.float32), np.zeros(2), 2),
                               bits=3, alphabet_scalar=4)
    assert np.array_equal(q._layer_alphabet(W), O.layer_alphabet(W, 4, O.unit_alphabet(3)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, axis, shape, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        full = np.arange(np.prod(shape), dtype=np.float64).reshape(shape) + 1.0
        net = hostnet.mnist_mlp(seed=1, widths=(6,), n_in=4, n_out=3)
        q = QuantizedNeuralNetwork(net, 1, hostnet.ArraySequence(np.zeros((1, 2, 2), np.float32), np.zeros(1), 1),
                                   shard=(rank, world))
        n = shape[axis]
        lo, hi = shard_range(n, rank, world)
        mine = np.zeros(shape)
        sl = [slice(None)] * len(shape)
        sl[axis] = slice(lo, hi)
        mine[tuple(sl)] = full[tuple(sl)]        # what this rank's C-ABI call would have written
        out = q._gather_columns(mine, lo, hi, axis)
        ret[rank] = bool(np.array_equal(out, full))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("axis,shape", [(1, (5, 7)), (2, (3, 3, 5, 4)), (1, (4, 1))])
def test_world2_gloo_gather_reassembles_q(axis, shape):
    """N > 1: every rank quantizes its shard of neurons / channels, Q blocks are all-gathered; no other collective."""
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_gather_worker, args=(r, world, port, axis, shape, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert dict(ret) == {0: True, 1: True}


def test_layerdata_same_detection():
    a = np.ones((3, 4), np.float32)
    assert LayerData(a, a).same and LayerData(a, a.copy()).same and not LayerData(a, a * 2).same


def _replicate_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from quantized_neural_networks_b200.replicate import h2d_bytes_per_rank, replicate_leading_axis
        ok = True
        for shape in [(7, 3), (8, 2, 2, 3), (1, 5), (5008 // 16, 4)]:
            a = np.arange(np.prod(shape), dtype=np.float32).reshape(shape) + 1
            t = replicate_leading_axis(a, rank, world)          # CPU tensors under gloo: same slicing / padding logic
            ok = ok and np.array_equal(t.numpy(), a)
            ok = ok and h2d_bytes_per_rank(shape, 4, world) * world >= a.nbytes
        ret[rank] = ok
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_input_replication_all_gather(world):
    """N > 1 input replication (SURVEY.md 8e item 1): each rank contributes 1 / world of the leading axis, one all-gather
    completes the array on every rank -- ragged and tiny leading axes included."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_replicate_worker, args=(r, world, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert dict(ret) == {r: True for r in range(world)}


class _NumpyGramEngine:
    """Test-only stand-in for GpfqEngine.gram_matrices: fp64 NumPy Grams of the samples it is handed (CPU tensors)."""

    def gram_matrices(self, X, Xq=None, sync=True, device_out=False):
        assert device_out and X.dtype == np.float32
        x = X.astype(np.float64)
        q = x if Xq is None else Xq.astype(np.float64)
        G2 = q @ q.T
        return (G2 if Xq is None else q @ x.T), G2


def _split_gram_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from quantized_neural_networks_b200.replicate import sample_split_gram
        ok = True
        rng = np.random.default_rng(11)
        for N0, m, same in [(5, 13, False), (4, 8, True), (3, 1, False), (6, 2, True), (7, 101, False)]:
            X = rng.standard_normal((N0, m)).astype(np.float32)
            Xq = X if same else (X + 0.1 * rng.standard_normal((N0, m))).astype(np.float32)
            G1, G2 = sample_split_gram(_NumpyGramEngine(), X, None if same else Xq, rank, world)
            x, q = X.astype(np.float64), Xq.astype(np.float64)
            ok = ok and np.allclose(G2.numpy(), q @ q.T, rtol=1e-13, atol=1e-13)
            ok = ok and np.allclose(G1.numpy(), q @ x.T, rtol=1e-13, atol=1e-13)
            ok = ok and ((G1 is G2) == same)
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_sample_split_gram_all_reduce(world):
    """N > 1 sample-split Gram stage (SURVEY.md 8e item 4): each rank contracts m / world samples, one all-reduce per
    matrix gives every rank the whole-sample Grams -- ragged sample counts and fewer samples than ranks included."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_split_gram_worker, args=(r, world, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert dict(ret) == {r: True for r in range(world)}


def test_prefer_sample_split_rule():
    from quantized_neural_networks_b200.replicate import prefer_sample_split
    assert not prefer_sample_split(784, 25000, 1)
    assert prefer_sample_split(784, 25000, 8)            # MNIST layer: 16 N0^2 = 9.8 MB against 8 N0 m = 157 MB
    assert not prefer_sample_split(25088, 1504, 8)       # VGG fc1: the Grams would be 10 GB, the inputs 0.3 GB
    assert prefer_sample_split(16384, 4_000_000, 2)      # inputs beyond one GPU's HBM: split regardless
    with pytest.raises(ValueError):
        QuantizedNeuralNetwork(hostnet.mnist_mlp(seed=1, widths=(6,), n_in=4, n_out=3), 1,
                               hostnet.ArraySequence(np.zeros((1, 2, 2), np.float32), np.zeros(1), 1), gram_split="rows")


class _NumpyConvGramEngine:
    """Test-only stand-in for GpfqEngine.conv_gram_nhwc: fp64 NumPy Grams of the oracle's patch matrices."""

    device = None

    def conv_gram_nhwc(self, act, actq, kernel_size=(3, 3), strides=(1, 1), padding="SAME", rate=(1, 1), c0=0, n_channels=None):
        actq = act if actq is None else actq
        C, kk = act.shape[3], kernel_size[0] * kernel_size[1]
        g = np.zeros((C, 2, kk, kk))
        for c in range(C):
            X = O.channel_patches(act, c, tuple(kernel_size), tuple(strides), padding, tuple(rate)).astype(np.float64)
            Xq = O.channel_patches(actq, c, tuple(kernel_size), tuple(strides), padding, tuple(rate)).astype(np.float64)
            g[c, 0], g[c, 1] = Xq @ X.T, Xq @ Xq.T
        return g


def _image_split_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from quantized_neural_networks_b200.replicate import image_split_conv_gram
        ok = True
        rng = np.random.default_rng(17)
        eng = _NumpyConvGramEngine()
        for n_img, H, Wd, C, same, pad in [(5, 6, 5, 3, False, "SAME"), (2, 4, 4, 2, True, "VALID"), (1, 5, 5, 2, False, "SAME")]:
            act = rng.standard_normal((n_img, H, Wd, C)).astype(np.float32)
            actq = act if same else (act + 0.1 * rng.standard_normal(act.shape)).astype(np.float32)
            g = image_split_conv_gram(eng, act, None if same else actq, (3, 3), (1, 1), pad, (1, 1), rank, world)
            full = eng.conv_gram_nhwc(act, actq, (3, 3), (1, 1), pad, (1, 1))
            ok = ok and np.allclose(g.numpy(), full, rtol=1e-12, atol=1e-12)
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_image_split_conv_gram_all_reduce(world):
    """N > 1 conv layers: every rank contracts n_img / world images of all channels, one all-reduce of the per-channel
    kk x kk Grams gives every rank the whole-batch matrices -- ragged image counts, fewer images than ranks."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_image_split_worker, args=(r, world, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert dict(ret) == {r: True for r in range(world)}


def test_grid_runner_host_logic_and_level_packing():
    """Grid enumeration in the driver's order, grouping of grid points with identical quantized inputs, int8 level packing."""
    from quantized_neural_networks_b200 import QuantizedCNNGrid, pack_levels, unpack_levels
    net = hostnet.cifar10_cnn(seed=2, size=8, widths=(2, 3, 4), dense=5, n_out=3)
    seq = hostnet.ArraySequence(np.zeros((4, 8, 8, 3), np.float32), np.zeros(4), 2)
    g = QuantizedCNNGrid(net, 2, seq, [np.log2(3), 2, 3, 4], [2, 3, 4, 5, 6])
    assert len(g.grid) == 20 and g.grid[0] == (np.log2(3), 2) and g.grid[1] == (np.log2(3), 3) and g.grid[-1] == (4, 6)
    assert [len(p.alphabet) for p in g.points][::5] == [3, 4, 8, 16] and g.q_train_size == 4
    a = np.arange(6, dtype=np.float32).reshape(2, 3)
    groups = g._groups([a, a.copy(), a + 1, a + 1, a], a)
    assert [(q is None, m) for q, m in groups] == [(True, [0, 1, 4]), (False, [2, 3])]
    A = 0.3 * np.linspace(-1, 1, 4)
    Q = np.array([[A[0], A[3], 0.0], [A[2], A[1], A[1]]])
    lev, A2 = pack_levels(Q, A)
    assert lev.tolist() == [[0, 3, -1], [2, 1, 1]] and np.array_equal(unpack_levels(lev, A2), Q)
    with pytest.raises(ValueError):
        pack_levels(np.array([0.123]), A)


def test_alphabets_above_64_levels_are_rejected_in_the_constructor():
    """GPFQ_MAX_K (include/gpfq.h): bits > 6 cannot run on the CUDA path; the mirror classes say so up front instead of
    failing at the first layer (the reference accepts any `bits`)."""
    import pytest
    from quantized_neural_networks_b200 import QuantizedCNN, QuantizedNeuralNetwork, hostnet
    net = hostnet.mnist_mlp(seed=0, widths=(8,), n_in=16, n_out=4)
    seq = hostnet.ArraySequence(np.zeros((4, 4, 4), np.float32), np.zeros(4, int), 2)
    for cls in (QuantizedNeuralNetwork, QuantizedCNN):
        with pytest.raises(ValueError, match="64 levels"):
            cls(net, 2, seq, bits=8)
        cls(net, 2, seq, bits=6)     # 64 levels: accepted
