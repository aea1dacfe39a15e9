"""TEST INFRASTRUCTURE ONLY -- per-channel alphabets stated with the literal C oracle.

Unit u (a Dense neuron, or the kernel slice W[:, :, ci, f] of a conv layer) with scale s_u walks with the levels
`np.float64(s_u) * A`: one correctly rounded fp64 product per level, which is what NumPy's `rad_u * alphabet` gives for a
float32 scalar rad_u.  Every decision is the reference's, made with those levels (`c_oracle.quantize_layer` on one column).
"""
from __future__ import annotations

import numpy as np

from . import c_oracle, gpfq_oracle as O


def unit_levels(A, s) -> np.ndarray:
    return np.float64(s) * np.asarray(A, dtype=np.float64)


def dense_layer(W, X, Xq, A, scales, cols=None) -> np.ndarray:
    """Neurons `cols` (default: all) of a (N0, N1) layer, neuron j against `scales[j] * A`; other columns stay 0."""
    W = np.ascontiguousarray(W, dtype=np.float32)
    Q = np.zeros(W.shape)
    for j in (range(W.shape[1]) if cols is None else cols):
        Q[:, j] = c_oracle.quantize_layer(W, X, Xq, unit_levels(A, scales[j]), j0=j, j1=j + 1)[:, j]
    return Q


def conv_layer(W, groups, patches, A, scales, c0=0, n_channels=None) -> np.ndarray:
    """Input channels c0 .. c0+n_channels-1 of a (kh, kw, C / groups, F) kernel: channel c walks the Fg filters of its group,
    the slice W[:, :, c % Cg, f] against `scales[c % Cg, f] * A`.  `patches(c) -> (Xp, Xqp)`, each (kh*kw, n)."""
    kh, kw, Cg, F = W.shape
    Fg = F // groups
    n_channels = Cg * groups - c0 if n_channels is None else n_channels
    Q = np.zeros(W.shape)
    for c in range(c0, c0 + n_channels):
        ci, f0 = c % Cg, (c // Cg) * Fg
        Xp, Xqp = patches(c)
        Wc = np.ascontiguousarray(W[:, :, ci, f0:f0 + Fg].reshape(kh * kw, Fg))
        Q[:, :, ci, f0:f0 + Fg] = dense_layer(Wc, Xp, Xqp, A, scales[ci, f0:f0 + Fg]).reshape(kh, kw, Fg)
    return Q


def msq(W, A, scales) -> np.ndarray:
    """Nearest level of every weight, W[..., u] against `scales[..., u] * A` (scales shaped like W's trailing axes)."""
    W = np.asarray(W, dtype=np.float32)
    s = np.broadcast_to(np.asarray(scales, dtype=np.float64), W.shape)
    out = np.empty(W.shape)
    for idx in np.ndindex(W.shape):
        out[idx] = O.bit_round(float(W[idx]), unit_levels(A, s[idx]))
    return out


class ChannelOracleEngine:
    """The engine's call surface (with `groups` and `scales`) routed through the C oracle; `scales=None` is the per-layer call."""
    last_stats = {}

    def dense_layer(self, X, Xq, W, A, j0=0, j1=None, method="auto", scales=None):
        Xq = X if Xq is None else Xq
        j1 = W.shape[1] if j1 is None else j1
        if scales is None:
            Q = np.zeros(W.shape)
            Q[:, j0:j1] = c_oracle.quantize_layer(np.ascontiguousarray(W[:, j0:j1]), X, Xq, A)
            return Q
        return dense_layer(W, X, Xq, A, scales, cols=range(j0, j1))

    def conv_channels(self, Xp, Xqp, W, A, c0=0, n_channels=None, scales=None):
        kh, kw, C, F = W.shape
        s = np.ones((C, F)) if scales is None else scales
        A0 = np.asarray(A, dtype=np.float64) if scales is not None else None
        Q = np.zeros(W.shape)
        for i in range(C):
            Wc = np.ascontiguousarray(W[:, :, i, :].reshape(kh * kw, F))
            Xqi = Xp[i] if Xqp is None else Xqp[i]
            if scales is None:
                Q[:, :, i, :] = c_oracle.quantize_layer(Wc, Xp[i], Xqi, A).reshape(kh, kw, F)
            else:
                Q[:, :, i, :] = dense_layer(Wc, Xp[i], Xqi, A0, s[i]).reshape(kh, kw, F)
        return Q

    def conv_layer_nhwc(self, act, actq, W, A, strides=(1, 1), padding="SAME", rate=(1, 1), c0=0, n_channels=None, groups=1,
                        scales=None):
        actq = act if actq is None else actq
        ks = tuple(W.shape[:2])
        rate = tuple(rate) if rate else (1, 1)

        def patches(c):
            return (O.channel_patches(act, c, ks, tuple(strides), padding, rate),
                    O.channel_patches(actq, c, ks, tuple(strides), padding, rate))
        if scales is None:
            scales, A = np.ones(W.shape[2:]), np.asarray(A, dtype=np.float64)   # 1.0 * A is A, bit for bit
        return conv_layer(W, groups, patches, A, scales, c0, n_channels)
