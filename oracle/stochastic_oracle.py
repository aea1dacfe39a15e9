"""TEST INFRASTRUCTURE ONLY -- stochastic rounding (SPFQ) stated in NumPy and, for whole layers, with the C restatement
`stochastic_oracle.c`.

    splitmix64(x)       = the SplitMix64 finaliser of x + 0x9E3779B97F4A7C15 (mod 2^64)
    draw(seed, u, t)    = (splitmix64(splitmix64(seed ^ splitmix64(u)) ^ t) >> 11) * 2^-53
    stoc_round(v, A, r) = A[0] unless v > A[0] (NaN too); A[K-1] if v >= A[K-1]; else with k = max{i : A[i] <= v} and
                          p = (v - A[k]) / (A[k+1] - A[k]): A[k+1] if r < p else A[k]

Unit ids: a Dense neuron j; the conv slice W[:, :, ci, f] is unit ci * F + f (F all filters of the kernel); MSQ element i of the
flattened kernel.  Step ids: the direction, the tap r * kw + col, 0 for MSQ.  Per-unit scales give the levels fl(s_u * A[k]).
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

from . import gpfq_oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "stochastic_oracle.c")
_SO = os.path.join(_HERE, "libstochastic_oracle.so")
_lib = None


def splitmix64(x):
    """Element-wise on uint64 arrays (or one Python int, returned as an int)."""
    scalar = np.isscalar(x) and not isinstance(x, np.ndarray)
    z = np.asarray(x, dtype=np.uint64) if not scalar else np.array([int(x) & 0xFFFFFFFFFFFFFFFF], dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return int(z[0]) if scalar else z


def draw(seed, u, t):
    """Uniform draws in [0, 1): exact fp64 (53-bit integers times 2^-53), broadcast over u and t."""
    u = np.asarray(u, dtype=np.uint64)
    t = np.asarray(t, dtype=np.uint64)
    key = splitmix64(np.uint64(int(seed)) ^ splitmix64(u))
    return (splitmix64(key ^ t) >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def stoc_round(v, A, r):
    """The stochastic quantizer, element-wise over v and r (A ascending, one alphabet)."""
    A = np.asarray(A, dtype=np.float64)
    v = np.asarray(v, dtype=np.float64)
    r = np.broadcast_to(np.asarray(r, dtype=np.float64), v.shape)
    K = len(A)
    k = np.clip(np.searchsorted(A, v, side="right") - 1, 0, max(K - 2, 0))   # max{i : A[i] <= v}
    lo, hi = A[k], A[np.minimum(k + 1, K - 1)]
    with np.errstate(invalid="ignore", divide="ignore"):
        p = (v - lo) / (hi - lo)
    out = np.where(r < p, hi, lo)
    out = np.where(v >= A[-1], A[-1], out)
    return np.where(v > A[0], out, A[0])


def unit_levels(A, s) -> np.ndarray:
    return np.float64(s) * np.asarray(A, dtype=np.float64)


# --------------------------------------------------------------------------------------
# NumPy walk (the reference's dtype ladder, gpfq_oracle.quantize_neuron with the stochastic quantizer)
# --------------------------------------------------------------------------------------
def quantize_neuron(w, X, Xq, A, seed, unit):
    N0, m = X.shape
    u = np.zeros(m)
    q = np.zeros(N0)
    r = draw(seed, unit, np.arange(N0))
    for t in range(N0):
        nrm = O._norm(Xq[t, :], 2)
        if nrm < O.DEAD_NORM:
            q[t] = 0.0
        elif abs(np.dot(Xq[t, :], u)) < O.PERP_DOT:
            q[t] = stoc_round(w[t], A, r[t])
        else:
            q[t] = stoc_round(np.dot(Xq[t, :], u + w[t] * X[t, :]) / (nrm ** 2), A, r[t])
        u += w[t] * X[t, :] - q[t] * Xq[t, :]
    return q


def numpy_dense_layer(W, X, Xq, A, seed, scales=None, cols=None, u0=0):
    W = np.asarray(W, dtype=np.float32)
    Xq = X if Xq is None else Xq
    Q = np.zeros(W.shape)
    for j in (range(W.shape[1]) if cols is None else cols):
        Aj = A if scales is None else unit_levels(A, scales[j])
        Q[:, j] = quantize_neuron(W[:, j], X, Xq, Aj, seed, u0 + j)
    return Q


# --------------------------------------------------------------------------------------
# C walk
# --------------------------------------------------------------------------------------
def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
            subprocess.check_call(["gcc", "-O2", "-pthread", "-fPIC", "-shared", "-ffp-contract=off", "-Wall", "-o", _SO, _SRC,
                                   "-lm"])
        _lib = ctypes.CDLL(_SO)
        _lib.so_layer.restype = ctypes.c_int
        _lib.so_layer.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_long, ctypes.c_void_p, ctypes.c_long,
                                  ctypes.c_long, ctypes.c_long, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64,
                                  ctypes.c_long, ctypes.c_void_p, ctypes.c_long, ctypes.c_int]
        _lib.so_draw.restype = ctypes.c_double
        _lib.so_draw.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64]
        _lib.so_splitmix64.restype = ctypes.c_uint64
        _lib.so_splitmix64.argtypes = [ctypes.c_uint64]
        _lib.so_stoc_round.restype = ctypes.c_double
        _lib.so_stoc_round.argtypes = [ctypes.c_double, ctypes.c_void_p, ctypes.c_int, ctypes.c_double]
    return _lib


def dense_layer(W, X, Xq, A, seed, scales=None, j0=0, j1=None, u0=0, nthreads=None) -> np.ndarray:
    """Columns j0..j1-1 of a (N0, N1) layer by the C walk, column j as unit u0 + j (levels scales[j] * A when given)."""
    X = np.ascontiguousarray(X, dtype=np.float32)
    Xq = X if Xq is None else np.ascontiguousarray(Xq, dtype=np.float32)
    W = np.ascontiguousarray(W, dtype=np.float32)
    A = np.ascontiguousarray(A, dtype=np.float64)
    N0, m = X.shape
    N1 = W.shape[1]
    j1 = N1 if j1 is None else j1
    s = None if scales is None else np.ascontiguousarray(scales, dtype=np.float64).reshape(-1)
    Q = np.zeros((N0, N1))
    nthreads = nthreads or len(os.sched_getaffinity(0))
    rc = lib().so_layer(X.ctypes.data, Xq.ctypes.data, N0, m, W.ctypes.data, N1, j0, j1, A.ctypes.data, len(A),
                        None if s is None else s.ctypes.data, int(seed), int(u0), Q.ctypes.data, N1, nthreads)
    if rc:
        raise RuntimeError(f"so_layer failed rc={rc}")
    return Q


def conv_layer(W, groups, patches, A, seed, scales=None, c0=0, n_channels=None) -> np.ndarray:
    """Input channels c0 .. c0+n_channels-1 of a (kh, kw, C / groups, F) kernel: channel c walks the Fg filters of its group with
    its patches `patches(c) -> (Xp, Xqp)`; the slice W[:, :, c % Cg, f] is unit (c % Cg) * F + f."""
    kh, kw, Cg, F = W.shape
    Fg = F // groups
    n_channels = Cg * groups - c0 if n_channels is None else n_channels
    Q = np.zeros(W.shape)
    for c in range(c0, c0 + n_channels):
        ci, f0 = c % Cg, (c // Cg) * Fg
        Xp, Xqp = patches(c)
        Wc = np.ascontiguousarray(W[:, :, ci, f0:f0 + Fg].reshape(kh * kw, Fg))
        sc = None if scales is None else np.asarray(scales)[ci, f0:f0 + Fg]
        Q[:, :, ci, f0:f0 + Fg] = dense_layer(Wc, Xp, Xqp, A, seed, sc, u0=ci * F + f0).reshape(kh, kw, Fg)
    return Q


def msq(W, A, seed, scales=None) -> np.ndarray:
    """Every weight of W rounded stochastically, element i (C order) as unit i; levels scales[..., u] * A with scales shaped like W's
    trailing axes."""
    W = np.asarray(W, dtype=np.float32)
    v = W.astype(np.float64).reshape(-1)
    r = draw(seed, np.arange(v.size), 0)
    if scales is None:
        return stoc_round(v, A, r).reshape(W.shape)
    s = np.broadcast_to(np.asarray(scales, dtype=np.float64), W.shape).reshape(-1)
    out = np.empty(v.size)
    for i in range(v.size):
        out[i] = stoc_round(v[i], unit_levels(A, s[i]), r[i])
    return out.reshape(W.shape)


def _seed_list(seeds, n):
    if isinstance(seeds, (list, tuple, np.ndarray)):
        return [int(s) for s in seeds]
    return [int(seeds)] * n


class StochasticOracleEngine:
    """The engine's call surface (`seeds`, `scales`, `groups`) through the C stochastic walk; `seeds=None` is nearest rounding by the
    literal C oracle (channel_oracle.ChannelOracleEngine)."""
    last_stats = {}

    def __init__(self):
        from .channel_oracle import ChannelOracleEngine
        self._nearest = ChannelOracleEngine()

    @staticmethod
    def _alphabets(A):
        single = isinstance(A, np.ndarray) and A.ndim == 1
        return single, ([A] if single else list(A))

    def dense_layer(self, X, Xq, W, A, j0=0, j1=None, method="auto", scales=None, seeds=None):
        if seeds is None:
            return self._nearest.dense_layer(X, Xq, W, A, j0=j0, j1=j1, method=method, scales=scales)
        single, als = self._alphabets(A)
        sd = _seed_list(seeds, len(als))
        outs = []
        for a, Aa in enumerate(als):
            sc = None if scales is None else (np.asarray(scales)[a] if np.ndim(scales) == 2 else scales)
            outs.append(dense_layer(W, X, Xq, Aa, sd[a], sc, j0=j0, j1=j1))
        return outs[0] if single else np.stack(outs)

    def dense_layer_from_gram(self, *args, **kwargs):
        raise NotImplementedError("the oracle walks from the data, not from Gram matrices")

    def conv_channels(self, Xp, Xqp, W, A, c0=0, n_channels=None, scales=None, seeds=None):
        if seeds is None:
            return self._nearest.conv_channels(Xp, Xqp, W, A, c0=c0, n_channels=n_channels, scales=scales)
        kh, kw, C, F = W.shape
        n_channels = C - c0 if n_channels is None else n_channels

        def patches(c):
            i = c - c0
            return Xp[i], (Xp[i] if Xqp is None else Xqp[i])
        single, als = self._alphabets(A)
        sd = _seed_list(seeds, len(als))
        outs = [conv_layer(W, 1, patches, Aa, sd[a], None if scales is None else (np.asarray(scales)[a] if np.ndim(scales) == 3
                                                                                  else scales), c0, n_channels)
                for a, Aa in enumerate(als)]
        return outs[0] if single else np.stack(outs)

    def conv_layer_nhwc(self, act, actq, W, A, strides=(1, 1), padding="SAME", rate=(1, 1), c0=0, n_channels=None, groups=1,
                        scales=None, seeds=None):
        if seeds is None:
            return self._nearest.conv_layer_nhwc(act, actq, W, A, strides=strides, padding=padding, rate=rate, c0=c0,
                                                 n_channels=n_channels, groups=groups, scales=scales)
        actq = act if actq is None else actq
        ks = tuple(W.shape[:2])
        rate = tuple(rate) if rate else (1, 1)

        def patches(c):
            return (O.channel_patches(act, c, ks, tuple(strides), padding, rate),
                    O.channel_patches(actq, c, ks, tuple(strides), padding, rate))
        single, als = self._alphabets(A)
        sd = _seed_list(seeds, len(als))
        outs = [conv_layer(W, groups, patches, Aa, sd[a], None if scales is None else (np.asarray(scales)[a] if np.ndim(scales) == 3
                                                                                       else scales), c0, n_channels)
                for a, Aa in enumerate(als)]
        return outs[0] if single else np.stack(outs)

    def msq(self, W, A, scales=None, seeds=None):
        if seeds is None:
            from .channel_oracle import msq as scaled_msq
            return scaled_msq(W, A, np.ones(np.shape(W)[-1:]) if scales is None else scales)
        return msq(W, A, seeds, scales)
