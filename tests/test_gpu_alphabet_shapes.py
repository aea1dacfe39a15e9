"""GPU: every walk on alphabets off the linspace grid, against the literal oracles.

The kernels read an alphabet three ways: the literal scan of the levels; a windowed scan when every level lies within 1 % of a
step of an ascending grid; and, for alphabets on the symmetric grid -a + k 2a / (K - 1) (alphabet_on_symmetric_grid), the
tensor-core walk and the int8 residual form, which decide on the grid and carry the decisions as level indices.  The families
below sit on each side of those gates: exact linspace levels, levels inside the 1 % window but off the grid, just outside it, a
middle level a hair off 0, a ternary alphabet with an offset middle, asymmetric and non-uniform levels, and alphabets only
nearest rounding takes (descending, permuted, a repeated level, one level).  Off-grid alphabets must keep off the tensor-core
walk and the int8 residual form; grid alphabets must stay on them where they ran before.
"""
import functools

import numpy as np
import pytest

from conftest import glorot, hidden_pair
from oracle import c_oracle, channel_oracle as CO, gpfq_oracle as O, sparse_oracle as SP, stochastic_oracle as SO
from test_gpu_channel_alphabets import _scales
from test_gpu_parity import check
from test_gpu_sparse import _lambda
from test_gpu_stochastic import _conv

pytestmark = pytest.mark.gpu

SEED = 0x5EED_A1FA_BE75_0001
DEAD = 2                                  # dead directions at the top of every Dense layer
PRUNED = 2                                # an all-zero neuron


def _grid(K):
    return lambda rad: rad * np.linspace(-1, 1, K)


def _near(K, frac):
    """rad * linspace(-1, 1, K) with the interior levels moved by +-frac of a step (alternating); the ends stay exact."""
    def levels(rad):
        A = rad * np.linspace(-1, 1, K)
        A[1:-1] += np.where(np.arange(1, K - 1) % 2, frac, -frac) * (2 * rad / (K - 1))
        return A
    return levels


def _fixed(*levels):
    return lambda rad: rad * np.array(levels, dtype=np.float64)


# name: (alphabet_scalar, levels as a function of rad, on the symmetric grid)
FAMILIES = {f"grid_K{K}_c{c}": (c, _grid(K), True)
            for K, c in ((2, 1), (3, 2), (4, 3.7), (5, 1), (16, 2), (33, 3.7), (64, 1))}
FAMILIES.update({
    "near_0.5pct_K4": (2, _near(4, 0.005), False),            # inside the 1 % window of the equispaced flag
    "near_0.9pct_K7": (2, _near(7, 0.009), False),
    "near_0.5pct_K16": (3, _near(16, 0.005), False),
    "outside_1.5pct_K5": (2, _near(5, 0.015), False),         # just outside it: the literal scan
    # on the grid within 2^-40 a, but a middle level that is not 0 would come out of the fast walks as the literal 0.0
    "tiny_middle_K5": (2, _fixed(-1, -0.5, 1e-14, 0.5, 1), False),
    "ternary_offset_middle": (2, _fixed(-1, 0.005, 1), False),
    "asymmetric_K5": (2, lambda rad: rad * np.linspace(-1, 2, 5), False),
    "non_uniform_K9": (2, _fixed(-1, -1 / 2, -1 / 4, -1 / 8, 0, 1 / 8, 1 / 4, 1 / 2, 1), False),
    # nearest rounding only: not non-decreasing, or a single level
    "descending_K5": (2, lambda rad: rad * np.linspace(1, -1, 5), False),
    "permuted_ternary": (2, _fixed(0, -1, 1), False),
    "repeated_level": (2, _fixed(-1, 0, 0, 1), False),
    "single_level": (2, _fixed(1), False),
})
ASCENDING = [f for f in FAMILIES if not f.startswith(("descending", "permuted", "single"))]
ODD = [f for f in ASCENDING if len(FAMILIES[f][1](1.0)) % 2]


def _alphabet(family, W):
    c, levels, _ = FAMILIES[family]
    rad = c * np.median(np.abs(W.flatten()))            # fp32 median, as layer_alphabet and bench.make_alphabet
    return levels(rad)


# name: (N0, N1, m, method, options, stats.reserved & 3 for grid alphabets: bit 0 int8 residual form, bit 1 tensor-core walk)
DENSE = {
    "stream": (96, 45, 300, "stream", {}, 0),
    "stream_fast": (96, 45, 300, "stream_fast", {}, 0),
    "tile": (33, 70, 200, "gram", {}, 0),
    "pipe": (300, 131, 500, "gram", {"sweep_walk": 2}, 0),
    "gram_rows_default": (2304, 130, 1500, "gram", {}, 2),            # the tensor-core walk by size
    "tc_forced": (300, 131, 500, "gram", {"sweep_walk": 1, "sweep_outer": 1}, 2),
    "residual_fp64": (1100, 70, 160, "gram", {"sweep_outer": 2, "sweep_i8": 2}, 0),
    "residual": (1100, 70, 160, "gram", {"sweep_outer": 2}, 3),
    "residual_two_chains": (1100, 2100, 160, "gram", {"sweep_outer": 2}, 3),
}


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


@functools.lru_cache(maxsize=None)
def _layer(name):
    N0, N1, m = DENSE[name][:3]
    rng = np.random.default_rng(sum(map(ord, name)))
    X, Xq = hidden_pair(rng, N0, m)
    X[:DEAD] = Xq[:DEAD] = 0.0
    W = glorot(rng, N0, N1)
    W[:, PRUNED] = 0.0
    every = 97 if N1 > 200 else 9 if N0 >= 2048 else 1           # few oracle neurons where the layer is large
    cols = sorted(set(range(0, N1, every)) | {N1 - 1, PRUNED})
    return X, Xq, W, cols, _scales(rng, N1, zero_at=1) * float(np.median(np.abs(W)))


def _assert_levels(Q, levels_of):
    """Every live entry of column j is one of levels_of(j); the dead directions hold the literal 0."""
    assert not Q[:DEAD].any()
    for j in range(Q.shape[1]):
        assert np.isin(Q[DEAD:, j], levels_of(j)).all(), j


def _assert_walk(name, family, stats):
    want = DENSE[name][5] if FAMILIES[family][2] else 0
    assert stats["reserved"] & 3 == want, (name, family, stats)


@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("name", list(DENSE))
def test_dense_matches_the_oracle(engine, options, name, family):
    N0, N1, m, method, opts, _ = DENSE[name]
    X, Xq, W, cols, _ = _layer(name)
    A = _alphabet(family, W)
    options(**opts)
    Q = engine.dense_layer(X, Xq, W, A, method=method)
    stats = dict(engine.last_stats)
    _assert_levels(Q, lambda j: A)
    ref = c_oracle.quantize_layer(W[:, cols], X, Xq, A)
    check(Q[:, cols], ref, W[:, cols], X, Xq, exact=method == "stream")
    _assert_walk(name, family, stats)


OTHER_PATHS = [n for n in DENSE if n != "gram_rows_default"]


@pytest.mark.parametrize("family", ASCENDING)
@pytest.mark.parametrize("name", OTHER_PATHS)
def test_dense_stochastic_matches_the_oracle(engine, options, name, family):
    N0, N1, m, method, opts, _ = DENSE[name]
    X, Xq, W, cols, _ = _layer(name)
    A = _alphabet(family, W)
    options(**opts)
    Q = engine.dense_layer(X, Xq, W, A, method=method, seeds=SEED)
    stats = dict(engine.last_stats)
    _assert_levels(Q, lambda j: A)
    ref = np.stack([SO.dense_layer(W, X, Xq, A, SEED, j0=j, j1=j + 1)[:, j] for j in cols], axis=1)   # neuron j draws as unit j
    if method == "stream":
        assert np.array_equal(Q[:, cols], ref), (name, family)
    else:
        assert O.agreement(Q[:, cols], ref) >= 0.9999, (name, family)
    _assert_walk(name, family, stats)


@pytest.mark.parametrize("family", ODD)
@pytest.mark.parametrize("name", OTHER_PATHS)
def test_dense_l1_penalty_matches_the_oracle(engine, options, name, family):
    N0, N1, m, method, opts, _ = DENSE[name]
    X, Xq, W, cols, _ = _layer(name)
    A = _alphabet(family, W)
    lam = _lambda(Xq, A, 0.4)
    options(**opts)
    Q = engine.dense_layer(X, Xq, W, A, method=method, l1_penalty=lam)
    stats = dict(engine.last_stats)
    _assert_levels(Q, lambda j: A)
    ref = SP.dense_layer(W[:, cols], X, Xq, A, lam)
    if method == "stream":
        assert np.array_equal(Q[:, cols], ref), (name, family)
    else:
        assert O.agreement(Q[:, cols], ref) >= 0.9999, (name, family)
    _assert_walk(name, family, stats)


@pytest.mark.parametrize("family", ASCENDING)
@pytest.mark.parametrize("name", OTHER_PATHS)
def test_dense_per_channel_matches_the_oracle(engine, options, name, family):
    """Per-channel alphabets: the walk is chosen from the base alphabet, neuron j walks with fl(s_j * A[k]) (s_1 = 0)."""
    N0, N1, m, method, opts, _ = DENSE[name]
    X, Xq, W, cols, s = _layer(name)
    A = FAMILIES[family][1](1.0)
    options(**opts)
    Q = engine.dense_layer(X, Xq, W, A, method=method, scales=s)
    stats = dict(engine.last_stats)
    _assert_levels(Q, lambda j: CO.unit_levels(A, s[j]))
    assert not Q[:, 1].any()
    ref = CO.dense_layer(W, X, Xq, A, s, cols=cols)[:, cols]
    if method == "stream":
        assert np.array_equal(Q[:, cols], ref), (name, family)
    else:
        assert O.agreement(Q[:, cols], ref) >= 0.9999, (name, family)
    _assert_walk(name, family, stats)


@pytest.mark.parametrize("K", [2, 3, 4, 7, 16, 33, 64])
def test_project_alphabets_keep_the_fast_walks(engine, options, K):
    """Every alphabet the project builds -- c * median|W| * linspace(-1, 1, K) on an fp32 median, and the per-channel base
    linspace(-1, 1, K) -- takes the tensor-core walk and the int8 residual form when asked for, with the weights of sweep_pipe;
    the same alphabet moved 0.5 % of a step off the grid does not."""
    rng = np.random.default_rng(K)
    N0, N1, m = 160, 40, 96
    X, Xq = hidden_pair(rng, N0, m)
    for trial in range(2):
        W = glorot(rng, N0, N1) * np.float32(10.0 ** rng.uniform(-3, 1))
        s = _scales(rng, N1) * float(np.median(np.abs(W)))
        for c in (1, 2, 3, 3.7, 5):
            for A, kw in ((O.layer_alphabet(W, c, np.linspace(-1, 1, K)), {}), (np.linspace(-1, 1, K), {"scales": s})):
                options(sweep_walk=2, sweep_outer=1)
                ref = engine.dense_layer(X, Xq, W, A, method="gram", **kw)
                for opts, want in (({"sweep_walk": 1, "sweep_outer": 1}, 2), ({"sweep_walk": 0, "sweep_outer": 2}, 3)):
                    options(**opts)
                    Q = engine.dense_layer(X, Xq, W, A, method="gram", **kw)
                    assert engine.last_stats["reserved"] & 3 == want, (K, c, trial, kw.keys(), engine.last_stats)
                    assert O.agreement(Q, ref) >= 0.9999, (K, c, trial, kw.keys())
        if K > 2:
            off = _near(K, 0.005)(float(np.median(np.abs(W))) * 2)
            for opts in ({"sweep_walk": 1, "sweep_outer": 1}, {"sweep_walk": 0, "sweep_outer": 2}):
                options(**opts)
                engine.dense_layer(X, Xq, W, off, method="gram")
                assert engine.last_stats["reserved"] & 3 == 0, (K, opts, engine.last_stats)


CONV = ["3x3_c32_corr", "3x3_planes", "11x11"]


@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("name", CONV)
def test_conv_matches_the_oracle(engine, name, family):
    ks, geo, act, actq, W, _, s, groups, patches = _conv(name)
    A = _alphabet(family, W)
    Q = engine.conv_layer_nhwc(act, actq, W, A, **geo)
    assert np.array_equal(Q, c_oracle.quantize_conv_layer(W, patches, A)), (name, family)
    if family not in ASCENDING:
        return
    assert np.array_equal(engine.conv_layer_nhwc(act, actq, W, A, seeds=SEED, **geo), SO.conv_layer(W, groups, patches, A, SEED))
    base = FAMILIES[family][1](1.0)
    Qs = engine.conv_layer_nhwc(act, actq, W, base, scales=s, **geo)
    assert np.array_equal(Qs, CO.conv_layer(W, groups, patches, base, s)), (name, family)
    assert np.array_equal(engine.conv_layer_nhwc(act, actq, W, base, scales=s, seeds=SEED, **geo),
                          SO.conv_layer(W, groups, patches, base, SEED, s)), (name, family)


def _probe_values(A, rng):
    """The levels, the midpoints of the real levels and of the grid through the ends, one ulp and 1e-9 of a step either side
    of each, values beyond both ends, and seeded values over the range."""
    A = np.asarray(A, dtype=np.float64)
    lo, hi = float(A.min()), float(A.max())
    span = max(hi - lo, abs(hi), 1e-30)
    grid = np.linspace(A[0], A[-1], max(len(A), 2))
    mids = np.concatenate([(A[1:] + A[:-1]) / 2, (grid[1:] + grid[:-1]) / 2, grid])
    eps = 1e-9 * span / max(len(A) - 1, 1)
    v = np.concatenate([A, mids, np.nextafter(mids, -np.inf), np.nextafter(mids, np.inf), mids - eps, mids + eps,
                        [lo - span, hi + span, lo - 1e-9 * span, hi + 1e-9 * span, 0.0, -0.0],
                        rng.uniform(lo - 0.2 * span, hi + 0.2 * span, 20_000)])
    return v


@pytest.mark.parametrize("family", list(FAMILIES))
def test_bit_round_and_msq_match_numpy(engine, family):
    rng = np.random.default_rng(sum(map(ord, family)))
    A = FAMILIES[family][1](0.37)
    v = _probe_values(A, rng)
    nearest = lambda x: np.array([O.bit_round(t, A) for t in np.asarray(x, np.float64)])
    assert np.array_equal(engine.bit_round(v, A), nearest(v)), family
    W = v.astype(np.float32)
    assert np.array_equal(engine.msq(W, A), nearest(W)), family
    if family in ASCENDING:
        assert np.array_equal(engine.bit_round(v, A, seeds=SEED), SO.stoc_round(v, A, SO.draw(SEED, np.arange(v.size), 0)))
        assert np.array_equal(engine.msq(W, A, seeds=SEED), SO.msq(W, A, SEED))
