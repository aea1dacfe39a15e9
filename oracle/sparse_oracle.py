"""TEST INFRASTRUCTURE ONLY -- sparse GPFQ (the L1 penalty of gpfq_set_l1_penalty) stated in NumPy and, for whole layers, with
the C restatement `sparse_oracle.c`.

One greedy step (fp64, correctly rounded), with nrm, d and num as in gpfq_oracle.quantize_weight:

    q   = 0                                      if nrm < 1e-16
    den = fl(nrm * nrm)
    v   = w_t if |d| < 1e-10 else fl(num / den)
    tau = fl(lambda / den)
    v'  = 0 if |v| <= tau else fl(v - copysign(tau, v))
    q   = Q(v')    nearest (gpfq_oracle.bit_round) or stoc_round with draw(seed, u, t) (stochastic_oracle)

The shrink is this project's definition: it is applied in value space, so that the :86 guard branch is thresholded too.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

from . import gpfq_oracle as O
from . import stochastic_oracle as S

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "sparse_oracle.c")
_SO = os.path.join(_HERE, "libsparse_oracle.so")
_lib = None


def shrink(v, tau):
    """Soft thresholding in value space, element-wise: 0 where |v| <= tau, else v - copysign(tau, v) (NaN stays NaN)."""
    v = np.asarray(v, dtype=np.float64)
    tau = np.asarray(tau, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        return np.where(np.abs(v) <= tau, 0.0, v - np.copysign(tau, v))


def step_value(num, den, lam):
    """The main branch's shrunk value fl(fl(num / den) - copysign(fl(lam / den), .)), or 0."""
    return shrink(np.float64(num) / np.float64(den), np.float64(lam) / np.float64(den))


def quantize_neuron(w, X, Xq, A, lam, seed=None, unit=0):
    """The literal walk of one neuron with the penalty; `seed` None: nearest rounding, else stochastic with draw(seed, unit, t)."""
    N0, m = X.shape
    u = np.zeros(m)
    q = np.zeros(N0)
    r = None if seed is None else S.draw(seed, unit, np.arange(N0))
    for t in range(N0):
        nrm = O._norm(Xq[t, :], 2)
        if nrm < O.DEAD_NORM:
            q[t] = 0.0
        else:
            den = nrm * nrm
            d = np.dot(Xq[t, :], u)
            v = np.float64(w[t]) if abs(d) < O.PERP_DOT else np.dot(Xq[t, :], u + w[t] * X[t, :]) / den
            v = float(shrink(v, lam / den))
            q[t] = O.bit_round(v, A) if seed is None else float(S.stoc_round(v, A, r[t]))
        u += w[t] * X[t, :] - q[t] * Xq[t, :]
    return q


def numpy_dense_layer(W, X, Xq, A, lam, seed=None, scales=None, cols=None, u0=0):
    W = np.asarray(W, dtype=np.float32)
    Xq = X if Xq is None else Xq
    Q = np.zeros(W.shape)
    for j in (range(W.shape[1]) if cols is None else cols):
        Aj = A if scales is None else S.unit_levels(A, scales[j])
        Q[:, j] = quantize_neuron(W[:, j], X, Xq, Aj, lam, seed, u0 + j)
    return Q


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
            subprocess.check_call(["gcc", "-O2", "-pthread", "-fPIC", "-shared", "-ffp-contract=off", "-Wall", "-o", _SO, _SRC,
                                   "-lm"])
        _lib = ctypes.CDLL(_SO)
        _lib.sp_layer.restype = ctypes.c_int
        _lib.sp_layer.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_long, ctypes.c_void_p, ctypes.c_long,
                                  ctypes.c_long, ctypes.c_long, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_double,
                                  ctypes.c_int, ctypes.c_uint64, ctypes.c_long, ctypes.c_void_p, ctypes.c_long, ctypes.c_int]
        _lib.sp_shrink.restype = ctypes.c_double
        _lib.sp_shrink.argtypes = [ctypes.c_double, ctypes.c_double]
    return _lib


def dense_layer(W, X, Xq, A, lam, seed=None, scales=None, j0=0, j1=None, u0=0, nthreads=None) -> np.ndarray:
    """Columns j0..j1-1 of a (N0, N1) layer by the C walk with penalty `lam`; `seed` None: nearest rounding, else stochastic with
    column j as unit u0 + j.  Levels scales[j] * A when scales are given."""
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
    rc = lib().sp_layer(X.ctypes.data, Xq.ctypes.data, N0, m, W.ctypes.data, N1, j0, j1, A.ctypes.data, len(A),
                        None if s is None else s.ctypes.data, float(lam), 0 if seed is None else 1, 0 if seed is None else int(seed),
                        int(u0), Q.ctypes.data, N1, nthreads)
    if rc:
        raise RuntimeError(f"sp_layer failed rc={rc}")
    return Q


def conv_layer(W, groups, patches, A, lam, seed=None, scales=None, c0=0, n_channels=None) -> np.ndarray:
    """Input channels c0 .. c0+n_channels-1 of a (kh, kw, C / groups, F) kernel (as stochastic_oracle.conv_layer) with penalty `lam`."""
    kh, kw, Cg, F = W.shape
    Fg = F // groups
    n_channels = Cg * groups - c0 if n_channels is None else n_channels
    Q = np.zeros(W.shape)
    for c in range(c0, c0 + n_channels):
        ci, f0 = c % Cg, (c // Cg) * Fg
        Xp, Xqp = patches(c)
        Wc = np.ascontiguousarray(W[:, :, ci, f0:f0 + Fg].reshape(kh * kw, Fg))
        sc = None if scales is None else np.asarray(scales)[ci, f0:f0 + Fg]
        Q[:, :, ci, f0:f0 + Fg] = dense_layer(Wc, Xp, Xqp, A, lam, seed, sc, u0=ci * F + f0).reshape(kh, kw, Fg)
    return Q


def _per_alphabet(v, n):
    if isinstance(v, (list, tuple, np.ndarray)):
        return list(v)
    return [v] * n


class SparseOracleEngine:
    """The engine's call surface (`l1_penalty`, `seeds`, `scales`, `groups`) through the C sparse walk; `l1_penalty=None` is the
    walk without the penalty (stochastic_oracle.StochasticOracleEngine)."""
    last_stats = {}

    def __init__(self):
        self._plain = S.StochasticOracleEngine()

    @staticmethod
    def _alphabets(A):
        single = isinstance(A, np.ndarray) and A.ndim == 1
        return single, ([A] if single else list(A))

    @staticmethod
    def _scale(scales, a, ndim):
        return None if scales is None else (np.asarray(scales)[a] if np.ndim(scales) == ndim else scales)

    def dense_layer(self, X, Xq, W, A, j0=0, j1=None, method="auto", scales=None, seeds=None, l1_penalty=None):
        if l1_penalty is None:
            return self._plain.dense_layer(X, Xq, W, A, j0=j0, j1=j1, method=method, scales=scales, seeds=seeds)
        single, als = self._alphabets(A)
        lams, sds = _per_alphabet(l1_penalty, len(als)), _per_alphabet(seeds, len(als))
        outs = [dense_layer(W, X, Xq, Aa, lams[a], sds[a], self._scale(scales, a, 2), j0=j0, j1=j1) for a, Aa in enumerate(als)]
        return outs[0] if single else np.stack(outs)

    def dense_layer_from_gram(self, *args, **kwargs):
        raise NotImplementedError("the oracle walks from the data, not from Gram matrices")

    def conv_channels(self, Xp, Xqp, W, A, c0=0, n_channels=None, scales=None, seeds=None, l1_penalty=None):
        if l1_penalty is None:
            return self._plain.conv_channels(Xp, Xqp, W, A, c0=c0, n_channels=n_channels, scales=scales, seeds=seeds)
        kh, kw, C, F = W.shape
        n_channels = C - c0 if n_channels is None else n_channels

        def patches(c):
            i = c - c0
            return Xp[i], (Xp[i] if Xqp is None else Xqp[i])
        single, als = self._alphabets(A)
        lams, sds = _per_alphabet(l1_penalty, len(als)), _per_alphabet(seeds, len(als))
        outs = [conv_layer(W, 1, patches, Aa, lams[a], sds[a], self._scale(scales, a, 3), c0, n_channels) for a, Aa in enumerate(als)]
        return outs[0] if single else np.stack(outs)

    def conv_layer_nhwc(self, act, actq, W, A, strides=(1, 1), padding="SAME", rate=(1, 1), c0=0, n_channels=None, groups=1,
                        scales=None, seeds=None, l1_penalty=None):
        if l1_penalty is None:
            return self._plain.conv_layer_nhwc(act, actq, W, A, strides=strides, padding=padding, rate=rate, c0=c0,
                                               n_channels=n_channels, groups=groups, scales=scales, seeds=seeds)
        actq = act if actq is None else actq
        ks = tuple(W.shape[:2])
        rate = tuple(rate) if rate else (1, 1)

        def patches(c):
            return (O.channel_patches(act, c, ks, tuple(strides), padding, rate),
                    O.channel_patches(actq, c, ks, tuple(strides), padding, rate))
        single, als = self._alphabets(A)
        lams, sds = _per_alphabet(l1_penalty, len(als)), _per_alphabet(seeds, len(als))
        outs = [conv_layer(W, groups, patches, Aa, lams[a], sds[a], self._scale(scales, a, 3), c0, n_channels)
                for a, Aa in enumerate(als)]
        return outs[0] if single else np.stack(outs)

    def msq(self, W, A, scales=None, seeds=None):
        return self._plain.msq(W, A, scales=scales, seeds=seeds)
