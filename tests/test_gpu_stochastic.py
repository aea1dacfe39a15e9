"""GPU: stochastic rounding (SPFQ, gpfq_set_rounding) on every walk, against the C and NumPy restatements of
oracle/stochastic_oracle.py.  Unit ids are global (Dense neuron j; conv slice ci * F + f; MSQ element i), so shards, channel ranges,
conv paths and batched alphabets must all reproduce the whole-layer walk."""
from ctypes import POINTER, byref, c_double, c_int32, c_uint64, c_void_p

import numpy as np
import pytest

from conftest import glorot, golden, hidden_pair
from oracle import gpfq_oracle as O, stochastic_oracle as SO
from quantized_neural_networks_b200 import QuantizedCNN, QuantizedNeuralNetwork, _lib
from quantized_neural_networks_b200.grid import QuantizedCNNGrid
from quantized_neural_networks_b200.quantized_network import layer_seed
from test_gpu_channel_alphabets import CONV as CHANNEL_CONV, _scales
from test_host_channel_alphabets import QUIET, channel_cnn, mlp
from test_host_stochastic import _weights_equal, with_stochastic_oracle

pytestmark = pytest.mark.gpu

SEED = 0x1234_5678_9ABC_DEF0


@pytest.fixture
def options(engine):
    touched = []

    def set_(**kw):
        for k, v in kw.items():
            engine.set_option(k, v)
            touched.append(k)
    yield set_
    for k in touched:
        engine.set_option(k, 0)


def _edge_values(A, rng, n):
    """Seeded values over and beyond the alphabet, with every level, midpoints, the ends, NaN and +-inf."""
    lo, hi = float(A[0]), float(A[-1])
    v = rng.uniform(lo - 0.3 * (hi - lo), hi + 0.3 * (hi - lo), n)
    special = np.concatenate([A, (A[1:] + A[:-1]) / 2, np.nextafter(A, -np.inf), np.nextafter(A, np.inf),
                              [np.nan, np.inf, -np.inf, 0.0, -0.0, 1e300, -1e300]])
    v[:special.size] = special
    return v


@pytest.mark.parametrize("bits", [np.log2(3), 2, 4, 6])
def test_bit_round_and_msq_equal_numpy(engine, bits):
    rng = np.random.default_rng(int(10 * bits))
    A = 0.37 * O.unit_alphabet(bits)
    v = _edge_values(A, rng, 1_000_003)
    want = SO.stoc_round(v, A, SO.draw(SEED, np.arange(v.size), 0))
    got = engine.bit_round(v, A, seeds=SEED)
    assert np.array_equal(got, want, equal_nan=True)
    W = v[np.abs(v) < 1e30].astype(np.float32)
    assert np.array_equal(engine.msq(W, A, seeds=SEED), SO.msq(W, A, SEED))
    # unbiased inside the range: the mean of many roundings of one value is that value
    x = np.full(400_000, float(A[1]) * 0.41 + float(A[2]) * 0.59)
    q = engine.bit_round(x, A, seeds=7)
    assert abs(q.mean() - x[0]) < 5 * np.sqrt(q.var() / q.size)


def test_msq_scaled_equals_numpy(engine):
    rng = np.random.default_rng(4)
    A = O.unit_alphabet(3)
    for W in (rng.standard_normal((400, 13)).astype(np.float32), rng.standard_normal((3, 3, 4, 6)).astype(np.float32)):
        s = _scales(rng, W.shape[-1:] if W.ndim == 2 else W.shape[-2:], zero_at=0)
        Q = engine.msq(W, A, scales=s, seeds=99)
        assert np.array_equal(Q, SO.msq(W, A, 99, s))
        assert np.all(Q[..., 0] == 0.0) if W.ndim == 2 else np.all(Q[..., 0, 0] == 0.0)


# name: (N0, N1, m, bits, method, options, dead directions)
DENSE = {
    "stream_ternary": (96, 45, 300, np.log2(3), "stream", {}, 3),
    "stream_2bit": (96, 45, 300, 2, "stream", {}, 3),
    "stream_fast_4bit": (96, 45, 300, 4, "stream_fast", {}, 3),
    "stream_long_m": (40, 9, 9000, 2, "stream", {}, 2),
    "stream_fast_long_m_6bit": (40, 9, 9000, 6, "stream_fast", {}, 2),
    "tile_pipe_ternary": (300, 200, 500, np.log2(3), "gram", {"sweep_walk": 2}, 4),
    "tile_pipe_3bit": (300, 131, 500, 3, "gram", {"sweep_walk": 2}, 4),
    "tile_pipe_6bit": (300, 131, 500, 6, "gram", {"sweep_walk": 2}, 4),
    "tile_odd_N0": (33, 70, 200, 2, "gram", {}, 1),                        # sweep_tile_kernel
    "tile_many_neurons": (160, 2100, 200, 3, "gram", {"sweep_walk": 2}, 2),
    "gram_rows_outer1": (1100, 70, 160, np.log2(3), "gram", {"sweep_outer": 1}, 5),
    "residual_fp64": (1100, 70, 160, 2, "gram", {"sweep_outer": 2, "sweep_i8": 2}, 5),
    "residual_one_chain": (1100, 300, 160, np.log2(3), "gram", {"sweep_outer": 3}, 5),
    "residual_two_chains": (1100, 2100, 160, np.log2(3), "gram", {"sweep_outer": 2}, 5),
    "gram_dmma": (300, 100, 500, 4, "gram", {"gram_kernel": 1}, 3),
    "gram_i8": (300, 100, 500, 4, "gram", {"gram_kernel": 2}, 3),
    "auto_tc_shape": (2100, 64, 3000, np.log2(3), "gram", {"sweep_outer": 1}, 2),   # the tensor-core walk by size
    "tc_ternary": (300, 131, 500, np.log2(3), "gram", {"sweep_walk": 1, "sweep_outer": 1}, 4),
    "tc_2bit": (300, 131, 500, 2, "gram", {"sweep_walk": 1, "sweep_outer": 1}, 4),
    "tc_4bit": (300, 131, 500, 4, "gram", {"sweep_walk": 1, "sweep_outer": 1}, 4),
    "tc_6bit": (300, 131, 500, 6, "gram", {"sweep_walk": 1, "sweep_outer": 1}, 4),
    "residual_i8_ternary": (1100, 70, 160, np.log2(3), "gram", {"sweep_outer": 2, "sweep_i8": 1}, 5),
    "residual_i8_4bit": (1100, 70, 160, 4, "gram", {"sweep_outer": 2, "sweep_i8": 1}, 5),
}


@pytest.mark.parametrize("name", list(DENSE))
def test_dense_matches_the_oracle(engine, options, name):
    N0, N1, m, bits, method, opts, dead = DENSE[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    X, Xq = hidden_pair(rng, N0, m)
    X[:dead] = 0.0
    Xq[:dead] = 0.0
    W = glorot(rng, N0, N1)
    W[:, 2] = 0.0                                  # a pruned neuron
    A = float(np.median(np.abs(W))) * 2 * O.unit_alphabet(bits)
    options(**opts)
    Q = engine.dense_layer(X, Xq, W, A, method=method, seeds=SEED)
    st = dict(engine.last_stats)
    cols = list(range(N1)) if N1 <= 200 else list(range(0, N1, 97)) + [N1 - 1]
    ref = SO.dense_layer(W, X, Xq, A, SEED)
    if method == "stream":
        assert np.array_equal(Q[:, cols], ref[:, cols]), (name, st)       # the literal walk: exact
    else:
        assert O.agreement(Q[:, cols], ref[:, cols]) >= 0.9999, (name, st)
    Qn = engine.dense_layer(X, Xq, W, A, method=method)
    stn = dict(engine.last_stats)
    assert not np.array_equal(Q, Qn)
    for k in ("method", "gram_kernel", "reserved", "kernel_launches"):      # the kernels of the nearest call
        assert st[k] == stn[k], (k, st, stn)
    if name.startswith(("tc_", "auto_tc")):
        assert st["reserved"] & 2, st
    if name.startswith("residual_i8"):
        assert st["reserved"] & 3 == 3, st


@pytest.mark.parametrize("name", ["dense_first_ternary", "dense_hidden_grid", "ties_and_dead"])
def test_golden_dense_vectors(engine, options, name):
    g = golden(name)
    X = g["X"]
    Xq = g["Xq"] if "Xq" in g.files else None
    W = g["W"]
    A = float(np.median(np.abs(W))) * O.unit_alphabet(np.log2(3))
    ref = SO.dense_layer(W, X, X if Xq is None else Xq, A, 3)
    for method in ("stream", "stream_fast", "gram"):
        assert np.array_equal(engine.dense_layer(X, Xq, W, A, method=method, seeds=3), ref), method
    options(sweep_walk=1)
    for outer in (1, 2):                  # the tensor-core walk: Gram rows, carried residuals
        options(sweep_outer=outer)
        Q = engine.dense_layer(X, Xq, W, A, method="gram", seeds=3)
        assert engine.last_stats["reserved"] & 2, engine.last_stats
        assert np.array_equal(Q, ref), outer


@pytest.mark.parametrize("bits", [np.log2(3), 2, 3, 4, 6])
@pytest.mark.parametrize("scaled", [False, True])
def test_tensor_core_walk_equals_sweep_pipe(engine, options, bits, scaled):
    """The stochastic tensor-core walk against sweep_pipe / sweep_tile on the same Grams, bit for bit: several ranges, a neuron
    count off the 128 grid, dead directions, a pruned neuron and (scaled) a zero scale."""
    rng = np.random.default_rng(int(bits * 100) + scaled)
    N0, N1, m = 2300, 131, 900
    X, Xq = hidden_pair(rng, N0, m)
    X[:3] = Xq[:3] = 0.0
    W = glorot(rng, N0, N1)
    W[:, 5] = 0.0
    A = O.unit_alphabet(bits)
    kw = {"scales": _scales(rng, N1, zero_at=1) * float(np.median(np.abs(W)))} if scaled else {}
    if not scaled:
        A = A * float(np.median(np.abs(W))) * 2
    options(sweep_outer=1, sweep_walk=2)
    ref = engine.dense_layer(X, Xq, W, A, method="gram", seeds=SEED, **kw)
    assert engine.last_stats["reserved"] & 2 == 0
    options(sweep_walk=1)
    Q = engine.dense_layer(X, Xq, W, A, method="gram", seeds=SEED, **kw)
    assert engine.last_stats["reserved"] & 2
    assert np.array_equal(Q, ref)
    options(sweep_outer=2, sweep_i8=1)    # the carried-residual form: int8 contractions, then the tensor-core walk
    Qr = engine.dense_layer(X, Xq, W, A, method="gram", seeds=SEED, **kw)
    assert engine.last_stats["reserved"] & 3 == 3
    assert O.agreement(Qr, ref) >= 0.9999


def test_vgg_fc1_full_size(engine):
    """VGG16 fc1 (N0 = 25088, m = 1504: the residual form), 512 neurons; sampled neurons against the C walk."""
    rng = np.random.default_rng(31)
    N0, N1, m = 25088, 512, 1504
    X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    A = np.float32(3) * np.median(np.abs(W)) * O.unit_alphabet(np.log2(3))
    Q = engine.dense_layer(X, Xq, W, A, seeds=SEED)
    st = dict(engine.last_stats)
    assert st["gram_kernel"] == 3 and st["reserved"] & 3 == 3, st      # int8 contractions, tensor-core walk
    cols = [0, 1, 200, 511]
    ref = np.stack([SO.dense_layer(W, X, Xq, A, SEED, j0=c, j1=c + 1)[:, c] for c in cols], axis=1)
    assert O.agreement(Q[:, cols], ref) >= 0.9999


def test_shards_batches_scales_and_devices(engine):
    import torch
    rng = np.random.default_rng(9)
    N0, N1, m = 300, 90, 700
    X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    A = O.unit_alphabet(3)
    s = _scales(rng, N1, zero_at=7) * float(np.median(np.abs(W)))
    ref = SO.dense_layer(W, X, Xq, A, 5, s)
    for method in ("stream", "stream_fast", "gram"):
        Qs = np.zeros_like(ref)
        for j0, j1 in ((0, 31), (31, 64), (64, 90)):
            Qs[:, j0:j1] = engine.dense_layer(X, Xq, W, A, j0=j0, j1=j1, method=method, scales=s, seeds=5)[:, j0:j1]
        assert O.agreement(Qs, ref) >= 0.9999 and np.all(Qs[:, 7] == 0.0), method
        assert np.array_equal(Qs, engine.dense_layer(X, Xq, W, A, method=method, scales=s, seeds=5)), method
    G1, G2 = engine.gram_matrices(torch.from_numpy(X).cuda(), torch.from_numpy(Xq).cuda())
    Qg = engine.dense_layer(X, Xq, W, A, method="gram", scales=s, seeds=5)
    assert np.array_equal(engine.dense_layer_from_gram(G1, G2, W, A, scales=s, seeds=5), Qg)
    Qd = engine.dense_layer(torch.from_numpy(X).cuda(), torch.from_numpy(Xq).cuda(), torch.from_numpy(W).cuda(), A, method="gram",
                            scales=s, seeds=5)
    assert np.array_equal(Qd.cpu().numpy(), Qg)
    # batched alphabets with their own seeds equal single calls
    As = [O.unit_alphabet(b) for b in (np.log2(3), 2, 4)]
    for method in ("stream", "gram"):
        Qb = engine.dense_layer(X, Xq, W, As, method=method, seeds=[11, 12, 13])
        for a in range(3):
            assert np.array_equal(Qb[a], engine.dense_layer(X, Xq, W, As[a], method=method, seeds=11 + a)), (method, a)


def test_determinism_no_sync_and_mode_reset(engine):
    import torch
    rng = np.random.default_rng(12)
    N0, N1, m = 200, 64, 400
    X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    A = O.unit_alphabet(2) * float(np.median(np.abs(W)))
    near = engine.dense_layer(X, Xq, W, A, method="gram")
    a = engine.dense_layer(X, Xq, W, A, method="gram", seeds=1)
    assert np.array_equal(a, engine.dense_layer(X, Xq, W, A, method="gram", seeds=1))
    assert not np.array_equal(a, engine.dense_layer(X, Xq, W, A, method="gram", seeds=2))
    assert np.array_equal(near, engine.dense_layer(X, Xq, W, A, method="gram"))    # nearest again after stochastic calls
    from quantized_neural_networks_b200.engine import GpfqEngine
    with GpfqEngine(0) as fresh:
        assert np.array_equal(near, fresh.dense_layer(X, Xq, W, A, method="gram"))
    dX, dXq, dW = (torch.from_numpy(t).cuda() for t in (X, Xq, W))
    outs = [engine.dense_layer(dX, dXq, dW, A, method=meth, seeds=sd, sync=False) for meth, sd in
            (("gram", 1), ("gram", 2), ("stream", 1))]
    torch.cuda.synchronize()
    assert np.array_equal(outs[0].cpu().numpy(), a)
    assert np.array_equal(outs[1].cpu().numpy(), engine.dense_layer(X, Xq, W, A, method="gram", seeds=2))
    assert np.array_equal(outs[2].cpu().numpy(), engine.dense_layer(X, Xq, W, A, method="stream", seeds=1))


CONV = dict(CHANNEL_CONV)
CONV["11x11"] = ((11, 11), (1, 1), (1, 1), "SAME", (2, 14, 14), 3, 5, 1, 3)
CONV["3x3_planes"] = ((3, 3), (1, 1), (1, 1), "SAME", (4, 12, 12), 5, 9, 1, 2)


def _conv(name):
    ks, strides, rate, pad, (n_img, H, Wd), C, F, groups, bits = CONV[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    W = (rng.uniform(-1, 1, (*ks, C // groups, F)) * 0.4).astype(np.float32)
    s = _scales(rng, W.shape[2:], zero_at=(0, 1)) * float(np.median(np.abs(W)))
    geo = dict(strides=strides, padding=pad, rate=rate)
    patches = lambda c: (O.channel_patches(act, c, ks, **geo), O.channel_patches(actq, c, ks, **geo))
    return ks, geo, act, actq, W, float(np.median(np.abs(W))) * 2 * O.unit_alphabet(bits), s, groups, patches


@pytest.mark.parametrize("name", list(CONV))
def test_conv_matches_the_oracle_every_entry_path(engine, name):
    import torch
    ks, geo, act, actq, W, A, s, groups, patches = _conv(name)
    gk = {"groups": groups} if groups > 1 else {}
    ref = SO.conv_layer(W, groups, patches, A, 17)
    Q = engine.conv_layer_nhwc(act, actq, W, A, seeds=17, **geo, **gk)
    assert np.array_equal(Q, ref), name
    st = dict(engine.last_stats)
    engine.conv_layer_nhwc(act, actq, W, A, **geo, **gk)
    stn = dict(engine.last_stats)
    for k in ("method", "gram_kernel", "reserved", "kernel_launches"):
        assert st[k] == stn[k], (k, st, stn)
    cuda = lambda a: torch.from_numpy(a).cuda()
    Qd = engine.conv_layer_nhwc(cuda(act), cuda(actq), cuda(W), A, seeds=17, **geo, **gk).cpu().numpy()
    assert np.array_equal(Qd, ref), name
    C = act.shape[3]
    c0, n_ch = (1, C - 2) if groups == 1 else (W.shape[2] // 2, W.shape[2])   # a shard that crosses a group
    Qs = engine.conv_layer_nhwc(act, actq, W, A, seeds=17, c0=c0, n_channels=n_ch, **geo, **gk)
    assert np.array_equal(Qs, SO.conv_layer(W, groups, patches, A, 17, None, c0, n_ch)), name
    if groups == 1:
        Qc = engine.conv_channels([patches(c)[0] for c in range(C)], [patches(c)[1] for c in range(C)], W, A, seeds=17)
        assert np.array_equal(Qc, ref), name
    if ks[0] * ks[1] <= 128:
        n_img = act.shape[0]
        gram = (engine.conv_gram_nhwc(act[:n_img // 2], actq[:n_img // 2], ks, **geo)
                + engine.conv_gram_nhwc(act[n_img // 2:], actq[n_img // 2:], ks, **geo))
        assert np.array_equal(engine.conv_layer_from_gram(gram, W, A, seeds=17, **gk), ref), name
    # per-channel scales with a zero scale
    Qsc = engine.conv_layer_nhwc(act, actq, W, A, scales=s, seeds=17, **geo, **gk)
    assert np.array_equal(Qsc, SO.conv_layer(W, groups, patches, A, 17, s)), name
    assert np.all(Qsc[:, :, 0, 1] == 0.0)


def test_conv_batched_seeds_equal_single_calls(engine):
    ks, geo, act, actq, W, _, s, groups, patches = _conv("5x5")
    As = [O.unit_alphabet(b) for b in (np.log2(3), 2, 4)]
    Qb = engine.conv_layer_nhwc(act, actq, W, As, seeds=[4, 5, 6], **geo)
    for a in range(3):
        assert np.array_equal(Qb[a], engine.conv_layer_nhwc(act, actq, W, As[a], seeds=4 + a, **geo)), a


def test_bad_arguments(engine):
    rng = np.random.default_rng(2)
    X, Xq = hidden_pair(rng, 20, 50)
    W = glorot(rng, 20, 6)
    A = O.unit_alphabet(2)
    for bad in (-1, 2 ** 64, 1.5, "1", [1, 2], object()):
        with pytest.raises(ValueError):
            engine.dense_layer(X, Xq, W, A, seeds=bad)
    with pytest.raises(ValueError):
        engine.dense_layer(X, Xq, W, [A, A], seeds=[1])
    lib = _lib.lib()
    ctx = engine._ctx
    one = (c_uint64 * 1)(5)
    assert lib.gpfq_set_rounding(ctx, 2, one, 1) == 1
    assert lib.gpfq_set_rounding(ctx, 1, None, 1) == 1
    assert lib.gpfq_set_rounding(ctx, 1, one, 0) == 1
    Q = np.zeros((2, 20, 6))
    K = np.array([len(A), len(A)], np.int32)
    AA = np.concatenate([A, A])
    st = _lib.GpfqStats()
    engine._bind_stream(False)
    call = lambda levels, k, n: lib.gpfq_dense_layer(ctx, c_void_p(X.ctypes.data), c_void_p(Xq.ctypes.data), 50, 20, 50,
                                                      c_void_p(W.ctypes.data), 6, 6, 0, 6, levels.ctypes.data_as(POINTER(c_double)),
                                                      k.ctypes.data_as(POINTER(c_int32)), n, c_void_p(Q.ctypes.data), 6, 0, byref(st))
    try:
        assert lib.gpfq_set_rounding(ctx, 1, one, 1) == 0
        assert call(AA, K, 2) == 1                                       # more alphabets than seeds
        assert call(A[::-1].copy(), K[:1], 1) == 1                       # not non-decreasing
        assert call(np.array([-1.0, np.inf, 1.0, 2.0]), K[:1], 1) == 1   # not finite
        assert call(A, K[:1], 1) == 0
        assert lib.gpfq_msq(ctx, c_void_p(W.ctypes.data), W.size, A[::-1].copy().ctypes.data_as(POINTER(c_double)), len(A),
                            c_void_p(Q.ctypes.data), 0) == 1
    finally:
        lib.gpfq_set_rounding(ctx, 0, None, 0)
    assert call(A[::-1].copy(), K[:1], 1) == 0                           # nearest rounding takes any alphabet


def test_networks_and_grid_match_the_oracle_engine(engine):
    rng = np.random.default_rng(3)
    xm = rng.random((64, 20)).astype(np.float32)
    from quantized_neural_networks_b200 import hostnet
    seq = hostnet.ArraySequence(xm, rng.integers(0, 10, 64), 32)
    net = mlp()
    kw = dict(logger=QUIET, bits=2, alphabet_scalar=3, rounding="stochastic", seed=9)
    gpu = QuantizedNeuralNetwork(net, 32, seq, method="stream", **kw)
    ref = with_stochastic_oracle(QuantizedNeuralNetwork, net, 32, seq, **kw)
    gpu.quantize_network()
    ref.quantize_network()
    assert _weights_equal(gpu.quantized_net, ref.quantized_net)
    cnn = channel_cnn()
    xc = np.random.default_rng(8).random((16, 8, 8, 3)).astype(np.float32)
    seqc = hostnet.ArraySequence(xc, np.zeros(16), 8)
    for scope in ("layer", "channel"):
        ckw = dict(logger=QUIET, bits=3, alphabet_scalar=2, rounding="stochastic", seed=4, alphabet_scope=scope)
        mirror = with_stochastic_oracle(QuantizedCNN, cnn, 8, seqc, **ckw)
        mirror.quantize_network()
        for path in ("nhwc", "patches"):
            q = QuantizedCNN(cnn, 8, seqc, conv_path=path, **ckw)
            q.quantize_network()
            assert _weights_equal(q.quantized_net, mirror.quantized_net), (scope, path)
    grid = QuantizedCNNGrid(cnn, 8, seqc, [2, 3], [2, 3], logger=QUIET, rounding="stochastic", seed=40).quantize_network()
    for g, ((bits, c), p) in enumerate(zip(grid.grid, grid.points)):
        one = QuantizedCNN(cnn, 8, seqc, logger=QUIET, bits=bits, alphabet_scalar=c, rounding="stochastic", seed=40 + g)
        one.quantize_network()
        assert _weights_equal(p.quantized_net, one.quantized_net), g
    for g, (p, msq) in enumerate(zip(grid.points, grid.msq_networks())):
        W = cnn.layers[0].get_weights()[0]
        A, _ = p._levels(W, "Conv2D")
        assert np.array_equal(msq.layers[0].get_weights()[0], SO.msq(W, A, layer_seed(40 + g, 0)).astype(np.float32))
