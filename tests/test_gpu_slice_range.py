"""The int8 digit-slice kernels on inputs of wide dynamic range.

Three hot paths hold fp64 operands as five balanced base-256 int8 digits, rounded 38 bits below an exponent shared by a row:
the tcgen05 Gram stage (gram_i8.cu, one exponent per direction), the tensor-core range walk (sweep_tc.cu, one per Gram row
G2[t, tb : block start]) and the residual form's int8 contractions (slgemm_i8.cu).  A small entry next to a large one that shares
its exponent keeps fewer bits, so data whose rows all have the same norm and no outliers never shows the error.  This file states
the slicing exactly in NumPy (`slices`, `model_product`, `model_level`), pins that model on the CPU, compares the Gram stage with it
on outliers, spikes, lognormal tails, spread row norms, subnormal and huge rows and the level thresholds, and runs every walk on
layers whose direction norms spread over 10^+-1 .. 10^+-3 -- with some decisions placed on purpose between the walk's flag band and
the slicing error of its Q terms.
"""
import functools

import numpy as np
import pytest

from oracle import c_oracle, channel_oracle as CO, gpfq_oracle as O, sparse_oracle as SP, stochastic_oracle as SO

S = 5                     # digits per value
P_BITS = 8 * S - 2        # bits kept below 2^e
D_OF_LEVEL = {0: S + 1, 1: S + 2, 2: 2 * S}   # slice pairs k + l <= D kept at each level of i8_row_exponent_kernel
RATIO_NARROW, RATIO_MEDIUM = 12.0, 128.0
SEED = 0x5EED_51CE_0000_0003
R = 512                   # directions per range of the walks at these neuron counts (SWEEP_OUTER, stc::MAX_R)
NB = 32                   # directions per block of the tensor-core walk


# ---- the exact model of the slicing ------------------------------------------------------------------------------------
def slices(M, axis=1):
    """Balanced base-256 digits of M with one exponent per row (axis=1) or per column (axis=0), as i8_split_kernel,
    stc_prepare_kernel and sl_rowsplit make them: e from frexp of the row maximum (0 for an all-zero row), v = rint(x 2^(38 - e))
    (= __double2ll_rn), digits b_1 (most significant) .. b_5 with v = sum b_k 2^(8 (5 - k)).  Returns (digits (5, rows, cols)
    int64, e (rows,) int64), rows along `axis`."""
    M = np.asarray(M, np.float64)
    if axis == 0:
        M = M.T
    e = np.frexp(np.abs(M).max(axis=1))[1].astype(np.int64) if M.shape[1] else np.zeros(M.shape[0], np.int64)
    v = np.rint(np.ldexp(M, (P_BITS - e)[:, None])).astype(np.int64)
    digits = np.empty((S,) + M.shape, np.int64)
    for k in range(S - 1, -1, -1):
        dg = ((v + 128) & 255) - 128
        v = (v - dg) >> 8
        digits[k] = dg
    assert not v.any()
    return digits, e


def sliced(M, axis=1):
    """The values the digits stand for: rint(x 2^(38 - e)) 2^(e - 38)."""
    dg, e = slices(M, axis)
    v = sum(dg[k].astype(np.float64) * 2.0 ** (8 * (S - 1 - k)) for k in range(S))
    out = np.ldexp(v, (e - P_BITS)[:, None])
    return out.T if axis == 0 else out


def model_product(A, B, D):
    """A B^T from the digit slices of A and B (one exponent per row of each), keeping the digit pairs k + l <= D: every pair
    product an exact integer matmul, combined in extended precision and scaled by 2^(4 - 8 (k + l) + eA + eB).  Returns (value,
    sum of the absolute terms, sum of the absolute terms of the dropped pairs)."""
    dA, eA = slices(A)
    dB, eB = slices(B)
    fA, fB = dA.astype(np.float64), dB.astype(np.float64)   # |pair sums| < 2^53: exact in fp64
    aA, aB = np.abs(fA), np.abs(fB)
    val = np.zeros((A.shape[0], B.shape[0]), np.longdouble)
    absv = np.zeros_like(val)
    drop = np.zeros_like(val)
    for k in range(1, S + 1):
        for l in range(1, S + 1):
            sc = np.longdouble(2.0) ** (4 - 8 * (k + l))
            if k + l <= D:
                val += (fA[k - 1] @ fB[l - 1].T).astype(np.longdouble) * sc
                absv += (aA[k - 1] @ aB[l - 1].T).astype(np.longdouble) * sc
            else:
                drop += (aA[k - 1] @ aB[l - 1].T).astype(np.longdouble) * sc
    ex = (eA[:, None] + eB[None, :]).astype(np.int64)
    f = lambda x: np.ldexp(x.astype(np.float64), ex)
    return f(val), f(absv), f(drop)


def model_level(*Xs):
    """The level i8_row_exponent_kernel raises for a call: per row, top = 2^e nnz against 12 sum|x| (level 1) and 128 sum|x|
    (level 2) -- the max over every row of every operand; 3 for a non-finite input."""
    lvl = 0
    for X in Xs:
        a = np.abs(np.asarray(X, np.float32))
        if not np.isfinite(a).all():
            return 3
        e = np.frexp(a.max(axis=1).astype(np.float64))[1]
        nnz = (a > 0).sum(axis=1)
        s = a.astype(np.float64).sum(axis=1)
        top = np.ldexp(1.0, e) * nnz
        live = nnz > 0
        lvl = max(lvl, int(np.where(top > RATIO_MEDIUM * s, 2, np.where(top > RATIO_NARROW * s, 1, 0))[live].max(initial=0)))
    return lvl


# ---- the model on the CPU ----------------------------------------------------------------------------------------------
def test_model_digits_rebuild_the_rounded_values():
    rng = np.random.default_rng(1)
    M = rng.standard_normal((40, 70)) * np.exp(3 * rng.standard_normal((40, 70)))
    M[3] = 0.0
    dg, e = slices(M)
    assert dg.min() >= -128 and dg.max() <= 127 and e[3] == 0
    sl = sliced(M)
    assert not sl[3].any()
    # rounded at 2^(e - 39) of the row, and exactly rint of the scaled values
    assert np.all(np.abs(sl - M) <= np.ldexp(1.0, e - P_BITS - 1)[:, None])
    assert np.array_equal(np.ldexp(sl, (P_BITS - e)[:, None]), np.rint(np.ldexp(M, (P_BITS - e)[:, None])))
    assert np.array_equal(sliced(M.T, axis=0), sl.T)


def test_model_is_exact_on_integer_data():
    rng = np.random.default_rng(2)
    A = rng.integers(-255, 256, (33, 500)).astype(np.float64)
    B = rng.integers(0, 256, (21, 500)).astype(np.float64)
    for D in (6, 7, 10):
        val, _, _ = model_product(A, B, D)
        assert np.array_equal(val, A @ B.T), D


def test_model_with_every_pair_is_the_product_of_the_sliced_values():
    rng = np.random.default_rng(3)
    A = (rng.standard_normal((17, 90)) * np.exp(2 * rng.standard_normal((17, 90)))).astype(np.float32)
    B = (np.maximum(rng.standard_normal((13, 90)), 0) * 10.0 ** rng.uniform(-3, 3, (13, 1))).astype(np.float32)
    val, absv, drop = model_product(A, B, 10)
    assert not drop.any()
    # the exact product of the sliced values, in integers: v_A v_B^T 2^(eA + eB - 76)
    dA, eA = slices(A)
    dB, eB = slices(B)
    vA = sum(dA[k].astype(object) * 2 ** (8 * (S - 1 - k)) for k in range(S))
    vB = sum(dB[k].astype(object) * 2 ** (8 * (S - 1 - k)) for k in range(S))
    exact = vA.dot(vB.T)
    ref = np.array([[float(np.ldexp(float(exact[i, j]), int(eA[i] + eB[j] - 2 * P_BITS))) for j in range(B.shape[0])]
                    for i in range(A.shape[0])])
    assert np.all(np.abs(val - ref) <= 2.0 ** -52 * absv)
    # dropping pairs changes the result by at most the dropped absolute terms
    for D in (6, 7):
        vD, _, dD = model_product(A, B, D)
        assert np.all(np.abs(vD - val) <= dD * (1 + 2.0 ** -40) + 2.0 ** -50 * absv)


def _threshold_row(ratio, past):
    """A row whose 2^e nnz is exactly `ratio` sum|x| (e = 0, powers of two: every sum is exact), or one fp32 ulp past it."""
    if ratio == RATIO_NARROW:
        r = [0.5, 0.25, 0.125, 0.0625] + [2.0 ** -7] * 8               # nnz 12, sum 1
    else:
        r = [0.5] + [2.0 ** -7] * 63 + [2.0 ** -13] * 64                # nnz 128, sum 1
    r = np.array(r, np.float32)
    if past:
        r[-1] = np.nextafter(r[-1], np.float32(0))
    return r


@pytest.mark.parametrize("ratio", [RATIO_NARROW, RATIO_MEDIUM])
def test_model_level_at_the_thresholds(ratio):
    rng = np.random.default_rng(4)
    base = np.maximum(rng.standard_normal((6, 2048)), 0).astype(np.float32)
    assert model_level(base) == 0
    for past in (False, True):
        X = base.copy()
        r = _threshold_row(ratio, past)
        X[2] = 0
        X[2, rng.choice(2048, r.size, replace=False)] = r
        want = (1 if ratio == RATIO_NARROW else 2) if past else (0 if ratio == RATIO_NARROW else 1)
        assert model_level(X) == want, (ratio, past)
    assert model_level(np.zeros((3, 10), np.float32)) == 0
    assert model_level(np.array([[1.0, np.inf]], np.float32)) == 3


# ---- input families of the Gram stage ----------------------------------------------------------------------------------
def _relu(rng, n, m):
    return np.maximum(rng.standard_normal((n, m)), 0)


def _family(kind, N0, m):
    rng = np.random.default_rng(N0 * 131 + m + sum(map(ord, kind)))
    if kind == "spikes_distinct":          # one spike per row, each in its own sample
        X = np.abs(rng.standard_normal((N0, m))) * 1e-4
        X[np.arange(N0), rng.integers(0, m, N0)] = 50.0
    elif kind == "lognormal_1.5":
        X = _relu(rng, N0, m) * np.exp(1.5 * rng.standard_normal((N0, m)))
    elif kind == "lognormal_2.5":
        X = _relu(rng, N0, m) * np.exp(2.5 * rng.standard_normal((N0, m)))
    elif kind == "row_spread":             # row norms over 10^+-3, no outliers inside a row
        X = _relu(rng, N0, m) * 10.0 ** rng.uniform(-3, 3, (N0, 1))
    elif kind == "one_nonzero":            # rows with a single non-zero of any size, and zero rows
        X = np.zeros((N0, m))
        X[np.arange(N0), rng.integers(0, m, N0)] = 10.0 ** rng.uniform(-3, 3, N0) * rng.choice([-1, 1], N0)
        X[::7] = 0.0
    elif kind == "all_negative":           # every other row all negative
        X = rng.standard_normal((N0, m))
        X[::2] = -np.abs(X[::2])
    elif kind == "tiny":                   # rows near 2^-126, subnormal fp32 entries among them
        X = _relu(rng, N0, m) * 2.0 ** rng.uniform(-130, -120, (N0, 1))
    elif kind == "huge":                   # rows near 2^127
        X = rng.uniform(0, 1, (N0, m)) * 2.0 ** rng.uniform(120, 127, (N0, 1))
    elif kind.startswith("threshold"):     # plain rows plus rows at / one ulp past the 12 and 128 ratios
        X = _relu(rng, N0, m)
        ratio = RATIO_NARROW if "12" in kind else RATIO_MEDIUM
        for i in range(3, N0, 29):
            r = _threshold_row(ratio, kind.endswith("past"))
            X[i] = 0
            X[i, rng.choice(m, r.size, replace=False)] = r
    else:
        raise ValueError(kind)
    X = X.astype(np.float32)
    if kind.startswith("threshold"):
        return X, X.copy()
    Xq = (X * (1 + 0.02 * rng.standard_normal(X.shape))).astype(np.float32)
    return X, Xq


FAMILIES = ["spikes_distinct", "lognormal_1.5", "lognormal_2.5", "row_spread", "one_nonzero", "all_negative", "tiny", "huge",
            "threshold12_at", "threshold12_past", "threshold128_at", "threshold128_past"]
GRAM_CASES = [(k, 256, 2048) for k in FAMILIES] + [("lognormal_1.5", 255, 1000), ("row_spread", 257, 3001),
                                                   ("spikes_distinct", 130, 26112), ("lognormal_2.5", 130, 26113)]


class _opts:
    def __init__(self, engine, **kw):
        self.engine, self.kw = engine, kw

    def __enter__(self):
        for k, v in self.kw.items():
            self.engine.set_option(k, v)

    def __exit__(self, *exc):
        for k in self.kw:
            self.engine.set_option(k, 0)


def _lower(G):
    return G[np.tril_indices(G.shape[0])]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,N0,m", GRAM_CASES)
def test_gram_i8_equals_the_slice_model(engine, kind, N0, m):
    """gram_kernel = 2 against model_product with D forced to 6, 7 and 10 and with the kernel's own choice, which must be the D
    model_level predicts: within a few hundred ulp of the fp64 combination of the sum of absolute terms (the kernel adds one
    fp64 term per K chunk, digit-pair sum and K split), and bit for bit the forced run of the predicted D."""
    X, Xq = _family(kind, N0, m)
    runs = {}
    for D in (6, 7, 10, 0):
        with _opts(engine, gram_kernel=2, i8_pairs_d=D):
            G1, G2 = engine.gram_matrices(X, Xq)
        runs[D] = (_lower(G1), _lower(G2))
        if D == 0:
            continue
        for G, (A, B) in ((G2, (Xq, Xq)), (G1, (Xq, X))):
            val, absv, _ = model_product(A, B, D)
            err = np.abs(_lower(G) - _lower(val))
            tol = 2.0 ** -44 * _lower(absv)
            assert np.all(err <= tol), (kind, D, float(np.max(err / np.maximum(_lower(absv), 1e-300))))
    want = D_OF_LEVEL[model_level(X, Xq)]
    assert all(np.array_equal(a, b) for a, b in zip(runs[0], runs[want])), (kind, want)
    if kind.startswith("threshold"):   # the rows at the thresholds make the three D distinguishable
        assert sum(np.array_equal(runs[0][1], runs[D][1]) for D in (6, 7, 10)) == 1


@pytest.mark.gpu
@pytest.mark.parametrize("kind", FAMILIES)
def test_gram_i8_within_the_slicing_bound(engine, kind):
    """Against an extended-precision Gram, under the bound the arithmetic gives: the slice rounding 2^-39 (2^eA ||B_s||_1 +
    2^eB ||A_t||_1), the dropped digit pairs, and the fp64 combination -- at the D the kernel picks itself."""
    X, Xq = _family(kind, 256, 2048)
    with _opts(engine, gram_kernel=2):
        G1, G2 = engine.gram_matrices(X, Xq)
    D = D_OF_LEVEL[model_level(X, Xq)]
    for G, (A, B) in ((G2, (Xq, Xq)), (G1, (Xq, X))):
        Al, Bl = A.astype(np.longdouble), B.astype(np.longdouble)
        ref = (Al @ Bl.T).astype(np.float64)
        eA, eB = slices(A)[1], slices(B)[1]
        n1A, n1B = np.abs(A.astype(np.float64)).sum(1), np.abs(B.astype(np.float64)).sum(1)
        _, absv, drop = model_product(A, B, D)
        bound = (2.0 ** -39 * (np.ldexp(1.0, eA)[:, None] * n1B[None, :] + np.ldexp(1.0, eB)[None, :] * n1A[:, None]) * (1 + 2.0 ** -30)
                 + drop + 2.0 ** -44 * absv)
        err = np.abs(_lower(G) - _lower(ref))
        assert np.all(err <= _lower(bound)), (kind, float(np.max(err / _lower(bound))))


# ---- the walks on layers of spread direction norms -----------------------------------------------------------------------
def _spread_layer(k, N0, N1, m, seed):
    """Strongly correlated directions (a rank-48 mix plus noise, ReLU) with row norms scaled by 10^U(-k, k)."""
    rng = np.random.default_rng(seed)
    Z = rng.standard_normal((48, m))
    X = np.maximum(rng.standard_normal((N0, 48)) @ Z + 0.3 * rng.standard_normal((N0, m)), 0)
    X = (X * 10.0 ** rng.uniform(-k, k, (N0, 1))).astype(np.float32)
    Xq = (X * (1 + 0.02 * rng.standard_normal(X.shape))).astype(np.float32)
    W = (rng.uniform(-1, 1, (N0, N1)) * np.sqrt(6.0 / (N0 + N1))).astype(np.float32)
    return X, Xq, W


MODES = ["nearest", "stochastic", "l1", "scales"]


def _mode_args(mode, W, X, Xq, bits):
    """(alphabet, engine keywords, oracle of the layer)."""
    if mode == "scales":
        rng = np.random.default_rng(7)
        s = (10.0 ** rng.uniform(-0.5, 0.5, W.shape[1])).astype(np.float32).astype(np.float64) * float(np.median(np.abs(W)))
        A = O.unit_alphabet(bits) * 3
        return A, {"scales": s}, lambda: CO.dense_layer(W, X, Xq, A, s)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(bits))
    if mode == "nearest":
        return A, {}, lambda: c_oracle.quantize_layer(W, X, Xq, A)
    if mode == "stochastic":
        return A, {"seeds": SEED}, lambda: SO.dense_layer(W, X, Xq, A, SEED)
    lam = 0.3 * float(np.max(np.abs(A))) * float(np.median(np.sum(np.asarray(Xq, np.float64) ** 2, axis=1)))
    return A, {"l1_penalty": lam}, lambda: SP.dense_layer(W, X, Xq, A, lam)


@functools.lru_cache(maxsize=None)
def _seeded(k):
    return _spread_layer(k, 1024, 48, 600, 100 + k)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("bits", [np.log2(3), 4], ids=["ternary", "16"])
@pytest.mark.parametrize("k", [1, 2, 3])
def test_walks_agree_on_spread_direction_norms(engine, k, bits, mode):
    """Row norms over 10^+-k: the tensor-core walk (Gram-row form) equals sweep_pipe bit for bit, the residual form's default
    takes the fp64 contractions (the spread gate) and equals sweep_i8 = 2 bit for bit, and every path agrees with the literal oracle on >= 99.99 % of the weights (the streaming walk
    exactly)."""
    X, Xq, W = _seeded(k)
    A, kw, oracle = _mode_args(mode, W, X, Xq, bits)
    ref = oracle()
    with _opts(engine, sweep_walk=1, sweep_outer=1):
        Qtc = engine.dense_layer(X, Xq, W, A, method="gram", **kw)
        assert engine.last_stats["reserved"] & 2
    with _opts(engine, sweep_walk=2, sweep_outer=1):
        Qpipe = engine.dense_layer(X, Xq, W, A, method="gram", **kw)
    with _opts(engine, sweep_outer=2):
        Qi8 = engine.dense_layer(X, Xq, W, A, method="gram", **kw)
        assert not engine.last_stats["reserved"] & 3   # past the spread gate of the int8 residual form: fp64 contractions
    with _opts(engine, sweep_outer=2, sweep_i8=2):
        Qf = engine.dense_layer(X, Xq, W, A, method="gram", **kw)
    Qs = engine.dense_layer(X, Xq, W, A, method="stream", **kw)
    assert np.array_equal(Qs, ref), int((Qs != ref).sum())
    assert np.array_equal(Qtc, Qpipe), int((Qtc != Qpipe).sum())
    for name, Q in (("tc", Qtc), ("pipe", Qpipe), ("residual_i8", Qi8), ("residual_fp64", Qf)):
        assert O.agreement(Q, ref) >= 0.9999, (name, O.agreement(Q, ref))
    assert np.array_equal(Qi8, Qf), int((Qi8 != Qf).sum())


# ---- adversarial placement: decisions between the flag band and the slicing error -------------------------------------
class _Quant:
    """The quantizer of one mode, stated literally: nearest rounding on the levels (per-channel: fl(s_j A)), stochastic rounding
    with the draw of (neuron j, step t), or nearest rounding of the value shrunk by tau = lambda / nrm^2.  `jumps` are the values
    of v where the decision of neuron j at step t changes."""

    def __init__(self, mode, A, N1, lam=None, s=None):
        self.mode, self.A, self.lam = mode, np.asarray(A, np.float64), lam
        self.L = np.stack([CO.unit_levels(self.A, s[j]) for j in range(N1)]) if mode == "scales" else None

    def levels(self, j):
        return self.L[j] if self.L is not None else self.A

    def decide(self, t, v, nrm2, cols):
        cols = np.asarray(cols)
        if self.mode == "stochastic":
            return SO.stoc_round(v, self.A, SO.draw(SEED, cols, t))
        if self.mode == "l1":
            v = SP.shrink(v, self.lam / nrm2)
        L = self.L[cols] if self.L is not None else np.broadcast_to(self.A, (len(cols), len(self.A)))
        return L[np.arange(len(cols)), np.argmin(np.abs(L - np.asarray(v)[:, None]), axis=1)]

    def jumps(self, t, j, nrm2):
        L = self.levels(j)
        if self.mode == "stochastic":
            return L[:-1] + float(SO.draw(SEED, j, t)) * (L[1:] - L[:-1])
        mids = 0.5 * (L[1:] + L[:-1])
        if self.mode == "l1":
            tau = self.lam / nrm2
            return np.where(mids > 0, mids + tau, mids - tau)
        return mids


def _place(W, G1, G2, quant, targets_of, delta_of):
    """Host pre-pass: the fp64 Gram-form walk (O.gram_quantize_layer's loop) with the mode's quantizer.  At the target step t_j
    of neuron j it takes d_t (extended precision; d_t does not depend on w_t) and picks the fp32 w_t whose exact value v lies
    delta_of(t, j) (signed, in steps of neuron j's levels) from the decision threshold nearest to the current v.  Returns the
    new weights, the decision each target must get, and the walk's decisions before the targets."""
    N0, N1 = W.shape
    Wd = W.astype(np.float64)
    Q = np.zeros((N0, N1))
    Wn = W.copy()
    want = {}
    cols = np.arange(N1)
    for t in range(N0):
        nrm = float(np.float32(np.sqrt(G2[t, t])))
        if nrm < O.DEAD_NORM:
            continue
        nrm2 = nrm ** 2
        d = G1[t, :t] @ Wd[:t] - G2[t, :t] @ Q[:t] if t else np.zeros(N1)
        for j in targets_of.get(t, ()):
            L = quant.levels(j)
            step = float(L[1] - L[0])
            if not step > 0:
                continue
            dl = (G1[t, :t].astype(np.longdouble) @ Wd[:t, j].astype(np.longdouble)
                  - G2[t, :t].astype(np.longdouble) @ Q[:t, j].astype(np.longdouble))
            if abs(float(dl)) < 1e3 * O.PERP_DOT:
                continue
            den = np.longdouble(nrm) ** 2
            v0 = float((dl + np.longdouble(Wd[t, j]) * np.longdouble(G1[t, t])) / den)
            thr = quant.jumps(t, j, nrm2)
            th = float(thr[np.argmin(np.abs(thr - v0))])
            delta = delta_of(t, j)
            w = np.float32(float((np.longdouble(th + delta * step) * den - dl) / np.longdouble(G1[t, t])))
            for _ in range(8):   # the fp32 rounding of w may cross the threshold: walk w by ulps to the wanted side
                v = (dl + np.longdouble(float(w)) * np.longdouble(G1[t, t])) / den
                off = float(v - np.longdouble(th)) / step
                if np.sign(off) == np.sign(delta) and abs(off) >= 2.0 ** -25:
                    break
                w = np.nextafter(w, np.float32(np.sign(delta) * np.sign(G1[t, t]) * np.inf))
            else:
                continue
            Wn[t, j] = w
            want[(t, j)] = float(quant.decide(t, np.array([float(v)]), nrm2, [j])[0])
        val = (d + Wd[t] * G1[t, t]) / nrm2
        val = np.where(np.abs(d) < O.PERP_DOT, Wd[t], val)
        Q[t] = quant.decide(t, val, nrm2, cols)
    return Wn, want, Q


def _lower_full(G):
    """A full matrix from the lower triangle the Gram stage leaves (G2 symmetric)."""
    L = np.tril(G)
    return L + np.tril(L, -1).T


def _slicing_error_of_p(G2, Q, t):
    """What the tensor-core walk's Q terms get wrong at step t for every neuron, in units of p: the rounding of the digit
    slices of G2[t, tb : t0] (one exponent for the row), times the range's decisions, over nrm_t^2."""
    tb, t0 = (t // R) * R, (t // NB) * NB
    if t0 <= tb:
        return np.zeros(Q.shape[1])
    g = G2[t, tb:t0][None, :]
    nrm2 = float(np.float32(np.sqrt(G2[t, t]))) ** 2
    return -((sliced(g)[0] - g[0]) @ Q[tb:t0]) / nrm2


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("bits", [np.log2(3), 4], ids=["ternary", "16"])
@pytest.mark.parametrize("k", [2, 3])
def test_tensor_core_walk_decides_past_the_slicing_error(engine, k, bits, mode):
    """One target step per neuron in a late block of a range, its weight chosen so that the exact decision argument lies delta
    (2^-24 .. 2^-14 of a step: outside the walk's 2^-30 band for more than three levels, partly inside its ~2^-20 ternary window)
    from a decision threshold -- the rounding midpoint, the stochastic threshold of the step's draw, or the midpoint moved out by
    the L1 shrink -- on the side opposite to where the slicing of the Gram rows moves the tensor-core walk's p.  The DMMA Gram
    (gram_kernel = 1) keeps the Gram stage exact to fp64 rounding, and the pre-pass walks the Grams the GPU computed.  The
    tensor-core walk must equal sweep_pipe on the whole layer, and both must take the pre-pass's decision at every target whose
    earlier decisions they share."""
    N0, N1, m = 1024, 128, 700
    X, Xq, W = _spread_layer(k, N0, N1, m, 200 + k)
    A, kw, _ = _mode_args(mode, W, X, Xq, bits)
    quant = _Quant(mode, A, N1, lam=kw.get("l1_penalty"), s=kw.get("scales"))
    with _opts(engine, gram_kernel=1):
        G1, G2 = engine.gram_matrices(X, Xq)
    G1, G2 = np.tril(G1), _lower_full(G2)
    _, _, Q0 = _place(W, G1, G2, quant, {}, None)
    steps = np.array([float(quant.levels(j)[1] - quant.levels(j)[0]) for j in range(N1)])
    # per neuron: the late-block direction where the modelled slicing error of p is largest
    cand = [t for t in range(N0) if (t % R) >= R - 4 * NB]
    errs = np.stack([_slicing_error_of_p(G2, Q0, t) for t in cand]) / np.where(steps > 0, steps, np.inf)
    best = np.argmax(np.abs(errs), axis=0)
    targets, delta = {}, {}
    for j in range(N1):
        t = cand[best[j]]
        e = errs[best[j], j]
        targets.setdefault(t, []).append(j)
        delta[(t, j)] = -np.sign(e or 1.0) * float(np.clip(abs(e) / 2, 2.0 ** -24, 2.0 ** -14))
    Wn, want, Qh = _place(W, G1, G2, quant, targets, lambda t, j: delta[(t, j)])
    assert len(want) >= N1 * 3 // 4
    with _opts(engine, gram_kernel=1, sweep_walk=1, sweep_outer=1):
        Qtc = engine.dense_layer(X, Xq, Wn, A, method="gram", **kw)
        assert engine.last_stats["reserved"] & 2 and engine.last_stats["gram_kernel"] == 1
    with _opts(engine, gram_kernel=1, sweep_walk=2, sweep_outer=1):
        Qpipe = engine.dense_layer(X, Xq, Wn, A, method="gram", **kw)
    tgt = list(want)
    bad_tc = sum(Qtc[t, j] != Qpipe[t, j] for t, j in tgt)
    assert bad_tc == 0 and np.array_equal(Qtc, Qpipe), (f"tensor-core walk vs sweep_pipe: {bad_tc} of {len(tgt)} targets, "
                                                      f"{int((Qtc != Qpipe).sum())} entries")
    shared = [(t, j) for t, j in tgt if np.array_equal(Qpipe[:t, j], Qh[:t, j])]
    assert len(shared) >= len(tgt) * 9 // 10
    bad = [(t, j) for t, j in shared if Qpipe[t, j] != want[(t, j)]]
    assert not bad, f"{len(bad)} of {len(shared)} targets off the pre-pass's decision"


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [np.log2(3), 4], ids=["ternary", "16"])
@pytest.mark.parametrize("N1", [70, 2100])
def test_residual_form_on_spread_direction_norms(engine, N1, bits):
    """The residual form (sweep_outer = 2) on layers shaped like its other tests, row norms over 10^+-2, with targets placed
    2^-16 of a step from a threshold on the smallest-norm directions.  One exponent per sample cannot hold those directions
    (forced int8 contractions, sweep_i8 = 1, decided 3-4 ternary targets wrongly), so the default must route the layer past
    its spread gate to the fp64 contractions: the same weights as sweep_i8 = 2 on the whole layer, and the pre-pass's decision
    at the targets.  (With m = 160 << N0 and spread norms the Gram form itself leaves the literal walk on ~1 % of the weights:
    no oracle bar here.)"""
    N0, m = 1100, 160
    X, Xq, W = _spread_layer(2, N0, N1, m, 300 + N1)
    A = O.layer_alphabet(W, 3, O.unit_alphabet(bits))
    G1, G2 = O.gram_matrices(X, Xq)
    norms = np.sqrt(np.diag(G2))
    small = [t for t in np.argsort(norms) if t >= 64][:16]
    rng = np.random.default_rng(N1)
    cols = range(N1) if N1 <= 128 else rng.choice(N1, 128, replace=False)
    targets = {}
    for i, j in enumerate(cols):
        targets.setdefault(int(small[i % len(small)]), []).append(int(j))
    sgn = {(t, j): float(rng.choice([-1, 1])) for t, js in targets.items() for j in js}
    Wn, want, Qh = _place(W, G1, G2, _Quant("nearest", A, N1), targets, lambda t, j: sgn[(t, j)] * 2.0 ** -16)
    runs = {}
    for i8 in (0, 2):
        with _opts(engine, sweep_outer=2, sweep_i8=i8):
            runs[i8] = engine.dense_layer(X, Xq, Wn, A, method="gram")
            assert engine.last_stats["gram_kernel"] == 3 and not engine.last_stats["reserved"] & 3
    tgt = list(want)
    diff = sum(runs[0][t, j] != runs[2][t, j] for t, j in tgt)
    assert diff == 0 and np.array_equal(runs[0], runs[2]), (diff, int((runs[0] != runs[2]).sum()))
    shared = [(t, j) for t, j in tgt if np.array_equal(runs[2][:t, j], Qh[:t, j])]
    assert len(shared) >= len(tgt) * 9 // 10
    bad = [(t, j) for t, j in shared if runs[2][t, j] != want[(t, j)]]
    assert not bad, f"{len(bad)} of {len(shared)} targets off the pre-pass's decision"
