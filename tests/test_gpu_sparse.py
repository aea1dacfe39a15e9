"""GPU: sparse GPFQ (the L1 penalty, gpfq_set_l1_penalty) on every walk, against the C restatement of oracle/sparse_oracle.py.
lambda = 0 must reproduce the call without the penalty bit for bit, a huge lambda gives all zeros for an odd number of levels, and
the tensor-core walk must equal sweep_pipe bit for bit."""
import numpy as np
import pytest

from conftest import glorot, hidden_pair
from oracle import gpfq_oracle as O, sparse_oracle as SP
from quantized_neural_networks_b200 import QuantizedCNN
from test_gpu_channel_alphabets import CONV as CHANNEL_CONV, _conv, _scales
from test_host_channel_alphabets import QUIET, channel_cnn
from test_host_sparse import _cnn_data, _weights_equal, with_sparse_oracle

pytestmark = pytest.mark.gpu

SEED = 0x0DDB_A11C_0FFE_E123
STATS = ("method", "gram_kernel", "reserved", "kernel_launches")


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


def _lambda(Xq, A, frac):
    """A penalty whose tau is about `frac` of the alphabet's radius on a typical direction."""
    den = float(np.median(np.sum(np.asarray(Xq, np.float64) ** 2, axis=1)))
    return frac * float(np.max(np.abs(A))) * den


# name: (N0, N1, m, method, options)
DENSE = {
    "stream": (96, 45, 300, "stream", {}),
    "stream_fast": (96, 45, 300, "stream_fast", {}),
    "stream_long_m": (40, 9, 9000, "stream", {}),
    "tile": (33, 70, 200, "gram", {}),
    "pipe": (300, 131, 500, "gram", {"sweep_walk": 2}),
    "tc": (300, 131, 500, "gram", {"sweep_walk": 1, "sweep_outer": 1}),
    "gram_rows": (1100, 70, 160, "gram", {"sweep_outer": 1}),
    "residual_fp64": (1100, 70, 160, "gram", {"sweep_outer": 2, "sweep_i8": 2}),
    "residual_i8": (1100, 70, 160, "gram", {"sweep_outer": 2, "sweep_i8": 1}),
    "residual_two_chains": (1100, 2100, 160, "gram", {"sweep_outer": 2}),
}
LEVELS = [3, 5, 7, 16]


@pytest.mark.parametrize("K", LEVELS)
@pytest.mark.parametrize("name", list(DENSE))
def test_dense_matches_the_oracle(engine, options, name, K):
    N0, N1, m, method, opts = DENSE[name]
    rng = np.random.default_rng(sum(map(ord, name)) + K)
    X, Xq = hidden_pair(rng, N0, m)
    X[:2] = Xq[:2] = 0.0                         # dead directions
    W = glorot(rng, N0, N1)
    W[:, 2] = 0.0                                # a pruned neuron
    A = float(np.median(np.abs(W))) * 2 * np.linspace(-1, 1, K)
    options(**opts)
    Qoff = engine.dense_layer(X, Xq, W, A, method=method)
    st_off = {k: engine.last_stats[k] for k in STATS}
    Q0 = engine.dense_layer(X, Xq, W, A, method=method, l1_penalty=0.0)
    assert np.array_equal(Q0, Qoff), name
    assert {k: engine.last_stats[k] for k in STATS} == st_off
    cols = list(range(N1)) if N1 <= 200 else list(range(0, N1, 97)) + [N1 - 1]
    lam = _lambda(Xq, A, 0.4)
    Q = engine.dense_layer(X, Xq, W, A, method=method, l1_penalty=lam)
    assert {k: engine.last_stats[k] for k in STATS} == st_off
    ref = SP.dense_layer(W[:, cols], X, Xq, A, lam)
    if method == "stream":
        assert np.array_equal(Q[:, cols], ref), name
    else:
        assert O.agreement(Q[:, cols], ref) >= 0.9999, name
    if K % 2:
        assert np.mean(Q == 0.0) > np.mean(Qoff == 0.0)
        assert not engine.dense_layer(X, Xq, W, A, method=method, l1_penalty=1e300).any()


@pytest.mark.parametrize("K", [3, 7])
def test_tensor_core_walk_equals_sweep_pipe_near_the_shifted_thresholds(engine, options, K):
    """Weights built so that many steps land on or next to the shifted thresholds a / 2 + tau (and on +-tau): the flagged blocks
    replay literally, so the two walks agree bit for bit, nearest and stochastic."""
    rng = np.random.default_rng(K)
    N0, N1, m = 320, 256, 400
    X = np.abs(rng.standard_normal((N0, m))).astype(np.float32)
    Xq = X.copy()
    W = glorot(rng, N0, N1)
    A = 0.05 * np.linspace(-1, 1, K)
    h = float(A[-1] - A[-2]) / 2
    lam = _lambda(Xq, A, 0.3)
    den = np.sum(X.astype(np.float64) ** 2, axis=1)
    tau = lam / den
    # first layer: the step's value is w_t itself up to the residual, so put w_t on the thresholds
    picks = rng.integers(0, 4, (N0, N1))
    shift = np.where(picks == 0, tau[:, None] + h, np.where(picks == 1, tau[:, None], np.where(picks == 2, -tau[:, None] - h, 0.0)))
    W = np.where(picks < 3, shift, W).astype(np.float32)
    for seeds in (None, SEED):
        out = []
        for walk in (1, 2):
            options(sweep_walk=walk, sweep_outer=1)
            out.append(engine.dense_layer(X, None, W, A, method="gram", l1_penalty=lam, seeds=seeds))
            assert bool(engine.last_stats["reserved"] & 2) == (walk == 1)
        assert np.array_equal(out[0], out[1]), seeds


def test_dense_from_gram_shards_and_batched_penalties(engine):
    import torch
    rng = np.random.default_rng(3)
    N0, N1, m = 300, 100, 500
    X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    As = [float(np.median(np.abs(W))) * c * np.linspace(-1, 1, 5) for c in (1.0, 2.0, 3.0)]
    lams = [_lambda(Xq, As[0], f) for f in (0.0, 0.3, 0.8)]
    batched = engine.dense_layer(X, Xq, W, As, l1_penalty=lams)
    for a in range(3):
        assert np.array_equal(batched[a], engine.dense_layer(X, Xq, W, As[a], l1_penalty=lams[a]))
    s = _scales(np.random.default_rng(3), (N1,))
    whole = engine.dense_layer(X, Xq, W, As[1], l1_penalty=lams[1], seeds=SEED, scales=s)
    part = engine.dense_layer(X, Xq, W, As[1], j0=30, j1=71, l1_penalty=lams[1], seeds=SEED, scales=s)
    assert np.array_equal(part[:, 30:71], whole[:, 30:71])
    ref = SP.dense_layer(W, X, Xq, As[1], lams[1], SEED, s)
    assert O.agreement(whole, ref) >= 0.9999
    G1, G2 = engine.gram_matrices(torch.from_numpy(X).cuda(), torch.from_numpy(Xq).cuda())
    Qg = engine.dense_layer_from_gram(G1, G2, W, As[1], l1_penalty=lams[1], seeds=SEED, scales=s)
    assert O.agreement(Qg, ref) >= 0.9999
    # determinism of device calls without a synchronisation
    cuda = lambda a: torch.from_numpy(a).cuda()
    outs = [engine.dense_layer(cuda(X), cuda(Xq), cuda(W), As[1], l1_penalty=lams[1], sync=False).cpu().numpy() for _ in range(3)]
    torch.cuda.synchronize()
    assert all(np.array_equal(o, outs[0]) for o in outs)
    with pytest.raises(Exception):
        engine.dense_layer(X, Xq, W, As, l1_penalty=[1.0, 2.0])


@pytest.mark.parametrize("name", list(CHANNEL_CONV))
def test_conv_matches_the_oracle_every_entry_path(engine, name):
    ks, geo, act, actq, W, _, s, groups, patches = _conv(name)
    A = float(np.median(np.abs(W))) * 2 * np.linspace(-1, 1, 5)
    gk = {"groups": groups} if groups > 1 else {}
    Xq0 = patches(0)[1]
    lam = _lambda(Xq0, A, 0.4)
    for kw in ({}, {"seeds": SEED}, {"scales": s}, {"seeds": SEED, "scales": s}):
        ref = SP.conv_layer(W, groups, patches, A, lam, kw.get("seeds"), kw.get("scales"))
        Q = engine.conv_layer_nhwc(act, actq, W, A, l1_penalty=lam, **geo, **gk, **kw)
        assert np.array_equal(Q, ref), (name, kw)
        Qoff = engine.conv_layer_nhwc(act, actq, W, A, **geo, **gk, **kw)
        stats = {k: engine.last_stats[k] for k in STATS}
        assert np.array_equal(engine.conv_layer_nhwc(act, actq, W, A, l1_penalty=0.0, **geo, **gk, **kw), Qoff), (name, kw)
        assert {k: engine.last_stats[k] for k in STATS} == stats
        C = act.shape[3]
        if groups == 1:
            Qc = engine.conv_channels([patches(c)[0] for c in range(C)], [patches(c)[1] for c in range(C)], W, A, l1_penalty=lam,
                                      **kw)
            assert np.array_equal(Qc, ref), (name, kw)
        if ks[0] * ks[1] <= 128:
            n_img = act.shape[0]
            gram = (engine.conv_gram_nhwc(act[:n_img // 2], actq[:n_img // 2], ks, **geo)
                    + engine.conv_gram_nhwc(act[n_img // 2:], actq[n_img // 2:], ks, **geo))
            assert np.array_equal(engine.conv_layer_from_gram(gram, W, A, l1_penalty=lam, **gk, **kw), ref), (name, kw)
    assert not engine.conv_layer_nhwc(act, actq, W, A, l1_penalty=1e300, **geo, **gk).any()
    both = engine.conv_layer_nhwc(act, actq, W, [A, 2 * A], l1_penalty=[lam, 0.5 * lam], **geo, **gk)
    assert np.array_equal(both[1], engine.conv_layer_nhwc(act, actq, W, 2 * A, l1_penalty=0.5 * lam, **geo, **gk))


def test_quantized_cnn_matches_the_oracle_engine_layer_by_layer(engine):
    net, seq = channel_cnn(), _cnn_data()
    kw = dict(logger=QUIET, bits=np.log2(5), alphabet_scalar=3, l1_penalty=0.5)
    gpu = QuantizedCNN(net, 8, seq, **kw)
    gpu.quantize_network()
    ref = with_sparse_oracle(QuantizedCNN, net, 8, seq, **kw)
    ref.quantize_network()
    for la, lb in zip(gpu.quantized_net.layers, ref.quantized_net.layers):
        for wa, wb in zip(la.get_weights(), lb.get_weights()):
            assert O.agreement(wa, wb) >= 0.999
    off = QuantizedCNN(net, 8, seq, **dict(kw, l1_penalty=0.0))
    off.quantize_network()
    plain = QuantizedCNN(net, 8, seq, **dict(kw, l1_penalty=None))
    plain.quantize_network()
    assert _weights_equal(off.quantized_net, plain.quantized_net)
