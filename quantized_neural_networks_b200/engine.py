"""Python face of the C ABI: one `GpfqEngine` per GPU.  Accepts NumPy arrays (host pointers; copies
happen inside the library call) or CUDA torch tensors (device pointers; torch is only the buffer)."""
from __future__ import annotations

import contextlib
import ctypes
import numbers
from ctypes import POINTER, byref, c_double, c_int32, c_uint64, c_void_p

import numpy as np

from . import _lib

try:  # torch is optional plumbing (device buffers / streams)
    import torch
except Exception:  # pragma: no cover
    torch = None

_METHODS = {"auto": _lib.METHOD_AUTO, "stream": _lib.METHOD_STREAM, "gram": _lib.METHOD_GRAM,
            "stream_fast": _lib.METHOD_STREAM_FAST}

# Conv kernel sizes kh * kw with batched Gram and walk kernels (every size up to 128 taps, 11 x 11 included): the set of
# `conv_supported_kk` in csrc/conv.cu.  Only these have the Gram-only entry points (`conv_gram_nhwc`, `conv_layer_from_gram`)
# and so the image split of a multi-GPU job; larger kernels run one Dense problem per channel.
CONV_SUPPORTED_KK = frozenset(range(1, 129))


def _is_torch(x):
    return torch is not None and isinstance(x, torch.Tensor)


def _alph_args(alphabets):
    """One alphabet (1-D) or a list of alphabets -> (levels*, K*, n, list)."""
    if isinstance(alphabets, np.ndarray) and alphabets.ndim == 1:
        alphabets = [alphabets]
    als = [np.ascontiguousarray(a, dtype=np.float64).reshape(-1) for a in alphabets]
    flat = np.concatenate(als) if als else np.zeros(0)
    K = np.array([len(a) for a in als], dtype=np.int32)
    return flat, K, len(als), als


def _scale_args(scales, n_alph, unit_shape, name="scales"):
    """Per-unit scales (per-channel alphabets) -> a contiguous float64 host array of n_alph x prod(unit_shape), or None.
    Accepts one table of unit_shape (used by every alphabet) or n_alph of them, as a NumPy array or a tensor."""
    if scales is None:
        return None
    if _is_torch(scales):
        scales = scales.detach().cpu().numpy()
    s = np.asarray(scales, dtype=np.float64)
    unit_shape = tuple(int(v) for v in unit_shape)
    if s.shape == unit_shape:
        s = np.broadcast_to(s, (n_alph,) + unit_shape)
    elif s.shape != (n_alph,) + unit_shape:
        raise ValueError(f"{name}: shape {s.shape}, expected {unit_shape} or {(n_alph,) + unit_shape}")
    if not np.all(np.isfinite(s)) or np.any(s < 0):
        raise ValueError(f"{name}: every scale must be finite and >= 0")
    return np.ascontiguousarray(s)


def _seed_args(seeds, n_alph):
    """Stochastic-rounding seeds -> None (nearest rounding) or a list of n_alph ints in [0, 2^64).  Accepts None, one int (used by
    every alphabet) or a sequence of n_alph ints."""
    if seeds is None:
        return None
    if isinstance(seeds, numbers.Integral) and not isinstance(seeds, bool):
        seeds = [seeds] * n_alph
    elif isinstance(seeds, (list, tuple, np.ndarray)):
        seeds = list(np.asarray(seeds, dtype=object).reshape(-1)) if isinstance(seeds, np.ndarray) else list(seeds)
        if len(seeds) != n_alph:
            raise ValueError(f"seeds: {len(seeds)} seeds for {n_alph} alphabets")
    else:
        raise ValueError(f"seeds: expected None, an int or a sequence of {n_alph} ints, got {type(seeds).__name__}")
    out = []
    for v in seeds:
        if not isinstance(v, numbers.Integral) or isinstance(v, bool) or not 0 <= int(v) < 1 << 64:
            raise ValueError(f"seeds: {v!r} is not an int in [0, 2^64)")
        out.append(int(v))
    return out


def _l1_args(l1_penalty, n_alph):
    """L1 penalty -> None (off) or a list of n_alph floats, each finite and >= 0.  Accepts None, one number (used by every
    alphabet) or a sequence of n_alph numbers."""
    if l1_penalty is None:
        return None
    if isinstance(l1_penalty, numbers.Real) and not isinstance(l1_penalty, bool):
        vals = [l1_penalty] * n_alph
    elif isinstance(l1_penalty, (list, tuple, np.ndarray)):
        vals = list(np.asarray(l1_penalty, dtype=object).reshape(-1)) if isinstance(l1_penalty, np.ndarray) else list(l1_penalty)
        if len(vals) != n_alph:
            raise ValueError(f"l1_penalty: {len(vals)} penalties for {n_alph} alphabets")
    else:
        raise ValueError(f"l1_penalty: expected None, a number or a sequence of {n_alph} numbers, got {type(l1_penalty).__name__}")
    out = []
    for v in vals:
        if not isinstance(v, numbers.Real) or isinstance(v, bool) or not np.isfinite(float(v)) or float(v) < 0:
            raise ValueError(f"l1_penalty: {v!r} is not a finite number >= 0")
        out.append(float(v))
    return out


def _dptr(a):
    return a.ctypes.data_as(POINTER(c_double))


class GpfqEngine:
    """Owns a `gpfq_ctx` (include/gpfq.h).  Fails loudly when the library or an sm_100 GPU is absent."""

    def __init__(self, device: int = 0):
        self._lib = _lib.lib()
        self._ctx = c_void_p()
        self.device = int(device)
        rc = self._lib.gpfq_create(self.device, byref(self._ctx))
        if rc != 0:
            self._ctx = c_void_p()
            raise _lib.GpfqError(rc, f"gpfq_create(device={device}) failed -- libgpfq needs a B200-class (sm_100) GPU; "
                                     "there is no CPU fallback")
        self.last_stats = {}

    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._lib.gpfq_destroy(self._ctx)
            self._ctx = c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- helpers --------------------------------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            msg = self._lib.gpfq_last_error(self._ctx)
            raise _lib.GpfqError(rc, msg.decode() if msg else "")

    def trim(self):
        self._check(self._lib.gpfq_trim(self._ctx))

    def conv_partial_bytes(self) -> int:
        """Bytes of partial Gram workspace the last conv call asked for (0 for kernels above 128 taps)."""
        return int(self._lib.gpfq_conv_partial_bytes(self._ctx))

    def set_option(self, key: str, value: int):
        """A/B switches of include/gpfq.h (`gram_kernel`, `i8_pairs_d`, `conv_kernel`, `corr_*`, `sweep_outer`, `sweep_walk`,
        `sweep_i8`)."""
        self._check(self._lib.gpfq_set_option(self._ctx, key.encode(), int(value)))

    @contextlib.contextmanager
    def _rounding(self, seeds, n_alph):
        """Stochastic rounding with these seeds for the calls inside (seeds None: nearest rounding); nearest again afterwards."""
        sd = _seed_args(seeds, n_alph)
        if sd is None:
            yield
            return
        arr = (c_uint64 * len(sd))(*sd)
        self._check(self._lib.gpfq_set_rounding(self._ctx, _lib.ROUND_STOCHASTIC, arr, len(sd)))
        try:
            yield
        finally:
            self._lib.gpfq_set_rounding(self._ctx, _lib.ROUND_NEAREST, None, 0)

    @contextlib.contextmanager
    def _penalty(self, l1_penalty, n_alph):
        """The L1 penalty (sparse GPFQ) for the calls inside (None: off); off again afterwards."""
        lam = _l1_args(l1_penalty, n_alph)
        if lam is None:
            yield
            return
        arr = (c_double * len(lam))(*lam)
        self._check(self._lib.gpfq_set_l1_penalty(self._ctx, arr, len(lam)))
        try:
            yield
        finally:
            self._lib.gpfq_set_l1_penalty(self._ctx, None, 0)

    def _bind_stream(self, dev):
        """Device-tensor calls launch on torch's CURRENT stream: the tensors were produced there, so this is what
        orders our kernels after their producers (and lets torch.cuda.Event brackets time them).  Host-array
        calls use the library's own stream."""
        s = None
        if dev:
            # torch's default stream has handle 0, which the C ABI reads as "the library's own stream":
            # name the legacy default stream explicitly (cudaStreamLegacy == 0x1)
            s = torch.cuda.current_stream(self.device).cuda_stream or 1
        self._check(self._lib.gpfq_set_stream(self._ctx, c_void_p(s)))

    def query_stats(self, calls_back=0):
        """Stage times of an earlier (possibly GPFQ_NO_SYNC) call; synchronise first."""
        st = _lib.GpfqStats()
        self._check(self._lib.gpfq_query_stats(self._ctx, int(calls_back), byref(st)))
        return st.as_dict()

    @staticmethod
    def _f32(x, name):
        if _is_torch(x):
            if x.dtype != torch.float32 or not x.is_cuda:
                raise TypeError(f"{name}: torch tensors must be float32 CUDA tensors")
            return x
        return np.asarray(x, dtype=np.float32)

    @staticmethod
    def _rowmajor2d(x, name):
        """(ptr, ld) of a 2-D array whose rows are contiguous."""
        if _is_torch(x):
            if x.dim() != 2 or x.stride(1) != 1:
                raise ValueError(f"{name}: need a 2-D tensor with contiguous rows")
            return x.data_ptr(), (x.stride(0) if x.shape[0] > 1 else x.shape[1])
        if x.ndim != 2:
            raise ValueError(f"{name}: need a 2-D array")
        if x.strides[1] != x.itemsize or (x.shape[0] > 1 and x.strides[0] % x.itemsize):
            raise ValueError(f"{name}: rows must be contiguous")
        return x.ctypes.data, (x.strides[0] // x.itemsize if x.shape[0] > 1 else x.shape[1])

    # -- Dense ----------------------------------------------------------------------------------
    def dense_layer(self, X, Xq, W, alphabets, j0=0, j1=None, method="auto", out=None, sync=True, scales=None, seeds=None,
                    l1_penalty=None):
        """Quantize neurons j0..j1-1 of a Dense layer.  X, Xq: (N0, m) fp32 feature-major (Xq may be
        None or X itself for the first layer); W: (N0, N1) fp32.  Returns Q fp64 (N0, N1) -- or
        (n_alphabets, N0, N1) when a list of alphabets is given -- with only the shard's columns written.
        `scales` (per-channel alphabets): (N1,) or (n_alphabets, N1), finite and >= 0; neuron j then walks with the levels
        fl64(scales[j] * alphabet[k]).  `seeds`: None rounds to the nearest level (the reference); an int or one int per alphabet in
        [0, 2^64) rounds stochastically (SPFQ, include/gpfq.h), neuron j drawing as unit j whatever the shard.  `l1_penalty`
        (sparse GPFQ): None walks without it; a number or one number per alphabet, finite and >= 0, soft-thresholds the value of
        every greedy step by lambda / nrm^2 before it is quantized (include/gpfq.h; 0.0 runs the penalty's kernels and gives the
        weights of the call without it)."""
        flat, K, n_alph, als = _alph_args(alphabets)
        single = isinstance(alphabets, np.ndarray) and alphabets.ndim == 1
        X = self._f32(X, "X")
        same = Xq is None or Xq is X
        Xq = X if same else self._f32(Xq, "Xq")
        W = self._f32(W, "W")
        dev = _is_torch(X)
        if dev != _is_torch(W) or dev != _is_torch(Xq):
            raise TypeError("X, Xq and W must all be NumPy arrays or all be CUDA tensors")
        if not dev:
            X = np.ascontiguousarray(X)
            Xq = X if same else np.ascontiguousarray(Xq)
            if W.ndim != 2 or W.strides[1] != W.itemsize:
                W = np.ascontiguousarray(W)
        if tuple(Xq.shape) != tuple(X.shape):
            raise ValueError("X and Xq must have the same shape")
        N0, m = int(X.shape[0]), int(X.shape[1])
        if W.shape[0] != N0:
            raise ValueError(f"W has {W.shape[0]} rows, X has {N0} directions")
        N1 = int(W.shape[1])
        j1 = N1 if j1 is None else int(j1)
        px, ldx = self._rowmajor2d(X, "X")
        pq, ldq_x = (px, ldx) if same else self._rowmajor2d(Xq, "Xq")
        if ldq_x != ldx:
            raise ValueError("X and Xq must share a row stride")
        pw, ldw = self._rowmajor2d(W, "W")
        self._bind_stream(dev)
        flags = _METHODS[method]
        if dev:
            flags |= _lib.ALL_DEVICE
            if out is None:
                out = torch.zeros((n_alph, N0, N1), dtype=torch.float64, device=X.device)
            pout = out.data_ptr()
            if not sync:
                flags |= _lib.NO_SYNC
        else:
            if out is None:
                out = np.zeros((n_alph, N0, N1), dtype=np.float64)
            pout = out.ctypes.data
        sc = _scale_args(scales, n_alph, (N1,))
        st = _lib.GpfqStats()
        args = (self._ctx, c_void_p(px), c_void_p(pq), ldx, N0, m, c_void_p(pw), ldw, N1, int(j0), j1,
                flat.ctypes.data_as(POINTER(c_double)), K.ctypes.data_as(POINTER(c_int32)), n_alph, c_void_p(pout), N1, flags,
                byref(st))
        with self._rounding(seeds, n_alph), self._penalty(l1_penalty, n_alph):
            rc = self._lib.gpfq_dense_layer(*args) if sc is None else self._lib.gpfq_dense_layer_scaled(*args, _dptr(sc))
        self._check(rc)
        self.last_stats = st.as_dict()
        return out[0] if single else out

    def gram_matrices(self, X, Xq=None, sync=True, device_out=False):
        """The Gram stage alone: (G1, G2) fp64 (N0, N0), lower triangle + diagonal valid (G1 is G2 when Xq is X / None).
        NumPy in -> NumPy out (diagnostics).  CUDA tensors in, or NumPy in with `device_out=True` (rows may be strided
        views, e.g. a sample range `X[:, lo:hi]`: the library copies them with one pitched H2D transfer) -> CUDA tensors
        out, contracted in place: the per-rank part of a sample-split Gram stage, see `dense_layer_from_gram`."""
        if _is_torch(X) or device_out:
            dev = _is_torch(X)
            X = self._f32(X, "X")
            same = Xq is None or Xq is X
            Xq = X if same else self._f32(Xq, "Xq")
            if _is_torch(Xq) != dev:
                raise TypeError("X and Xq must both be NumPy arrays or both be CUDA tensors")
            if tuple(Xq.shape) != tuple(X.shape):
                raise ValueError("X and Xq must have the same shape")
            N0, m = int(X.shape[0]), int(X.shape[1])
            px, ldx = self._rowmajor2d(X, "X")
            pq, ldq_x = (px, ldx) if same else self._rowmajor2d(Xq, "Xq")
            if ldq_x != ldx:
                raise ValueError("X and Xq must share a row stride")
            tdev = X.device if dev else torch.device("cuda", self.device)
            G2 = torch.empty((N0, N0), dtype=torch.float64, device=tdev)
            G1 = G2 if same else torch.empty((N0, N0), dtype=torch.float64, device=tdev)
            self._bind_stream(True)
            flags = (_lib.X_DEVICE if dev else 0) | _lib.Q_DEVICE | (0 if sync or not dev else _lib.NO_SYNC)
            rc = self._lib.gpfq_gram_matrices(self._ctx, c_void_p(px), c_void_p(pq), ldx, N0, m,
                                              c_void_p(None if same else G1.data_ptr()), c_void_p(G2.data_ptr()), flags)
            self._check(rc)
            return G1, G2
        X = np.ascontiguousarray(X, dtype=np.float32)
        same = Xq is None or Xq is X
        Xq = X if same else np.ascontiguousarray(Xq, dtype=np.float32)
        N0, m = X.shape
        G2 = np.zeros((N0, N0))
        G1 = G2 if same else np.zeros((N0, N0))
        self._bind_stream(False)
        rc = self._lib.gpfq_gram_matrices(self._ctx, c_void_p(X.ctypes.data), c_void_p(Xq.ctypes.data), m, N0, m,
                                          c_void_p(None if same else G1.ctypes.data), c_void_p(G2.ctypes.data), 0)
        self._check(rc)
        return G1, G2

    def dense_layer_from_gram(self, G1, G2, W, alphabets, j0=0, j1=None, out=None, sync=True, scales=None, seeds=None,
                              l1_penalty=None):
        """Sweep stage of a Dense layer from (N0, N0) fp64 Gram matrices on the device (CUDA tensors; G1 None or G2
        itself for the first layer): what every rank of a sample-split job runs after the all-reduce of the partial
        Grams.  W: (N0, N1) fp32 NumPy array or CUDA tensor; the result follows W's kind.  `scales`, `seeds` and `l1_penalty`
        as in `dense_layer`."""
        flat, K, n_alph, als = _alph_args(alphabets)
        single = isinstance(alphabets, np.ndarray) and alphabets.ndim == 1
        if not _is_torch(G2) or G2.dtype != torch.float64 or not G2.is_cuda or not G2.is_contiguous():
            raise TypeError("G2 must be a contiguous float64 CUDA tensor")
        same = G1 is None or G1 is G2
        if not same and (not _is_torch(G1) or G1.dtype != torch.float64 or not G1.is_cuda or not G1.is_contiguous()
                         or tuple(G1.shape) != tuple(G2.shape)):
            raise TypeError("G1 must be a contiguous float64 CUDA tensor shaped like G2")
        N0 = int(G2.shape[0])
        if G2.dim() != 2 or int(G2.shape[1]) != N0:
            raise ValueError("G2 must be (N0, N0)")
        W = self._f32(W, "W")
        wdev = _is_torch(W)
        if not wdev and (W.ndim != 2 or W.strides[1] != W.itemsize):
            W = np.ascontiguousarray(W)
        if W.shape[0] != N0:
            raise ValueError(f"W has {W.shape[0]} rows, the Gram matrices have {N0}")
        N1 = int(W.shape[1])
        j1 = N1 if j1 is None else int(j1)
        pw, ldw = self._rowmajor2d(W, "W")
        self._bind_stream(True)
        flags = _lib.X_DEVICE
        if wdev:
            flags |= _lib.W_DEVICE | _lib.Q_DEVICE
            if out is None:
                out = torch.zeros((n_alph, N0, N1), dtype=torch.float64, device=W.device)
            pout = out.data_ptr()
            if not sync:
                flags |= _lib.NO_SYNC
        else:
            if out is None:
                out = np.zeros((n_alph, N0, N1), dtype=np.float64)
            pout = out.ctypes.data
        sc = _scale_args(scales, n_alph, (N1,))
        st = _lib.GpfqStats()
        args = (self._ctx, c_void_p(None if same else G1.data_ptr()), c_void_p(G2.data_ptr()), N0, c_void_p(pw), ldw, N1,
                int(j0), j1, flat.ctypes.data_as(POINTER(c_double)), K.ctypes.data_as(POINTER(c_int32)), n_alph,
                c_void_p(pout), N1, flags, byref(st))
        with self._rounding(seeds, n_alph), self._penalty(l1_penalty, n_alph):
            rc = (self._lib.gpfq_dense_layer_from_gram(*args) if sc is None
                  else self._lib.gpfq_dense_layer_from_gram_scaled(*args, _dptr(sc)))
        self._check(rc)
        self.last_stats = st.as_dict()
        return out[0] if single else out

    # -- Conv -----------------------------------------------------------------------------------
    def conv_channels(self, Xp, Xqp, W, alphabets, c0=0, n_channels=None, out=None, sync=True, scales=None, seeds=None,
                      l1_penalty=None):
        """Quantize channels c0..c0+n_channels-1 of a (kh, kw, C, F) kernel from per-channel patch
        matrices.  Xp/Xqp: sequences (len n_channels) of (kh*kw, n_patches) fp32 arrays/tensors, or one
        (n_channels, kh*kw, n_patches) array; Xqp None => first conv layer (X == Xq).  `scales` (per-channel alphabets):
        (C, F) or (n_alphabets, C, F), finite and >= 0; the slice W[:, :, c, f] walks with fl64(scales[c, f] * alphabet[k]).
        `seeds` as in `dense_layer`; the slice W[:, :, c, f] draws as unit c * F + f, tap r * kw + col as step.  `l1_penalty` as
        in `dense_layer`."""
        flat, K, n_alph, als = _alph_args(alphabets)
        single = isinstance(alphabets, np.ndarray) and alphabets.ndim == 1
        W = self._f32(W, "W")
        kh, kw, C, F = (int(v) for v in W.shape)
        kk = kh * kw
        n_channels = (C - c0) if n_channels is None else int(n_channels)
        xs = [self._f32(Xp[i], "Xp") for i in range(n_channels)]
        same = Xqp is None
        qs = xs if same else [self._f32(Xqp[i], "Xqp") for i in range(n_channels)]
        dev = _is_torch(W)
        if any(_is_torch(x) != dev for x in xs + qs):
            raise TypeError("patches and W must all be NumPy arrays or all be CUDA tensors")
        if not dev:
            xs = [np.ascontiguousarray(x) for x in xs]
            qs = xs if same else [np.ascontiguousarray(q) for q in qs]
            W = np.ascontiguousarray(W)
        else:
            if not W.is_contiguous() or any(not x.is_contiguous() for x in xs + qs):
                raise ValueError("device tensors must be contiguous")
        n = int(xs[0].shape[1]) if n_channels else 1
        for x in xs + qs:
            if tuple(x.shape) != (kk, n):
                raise ValueError(f"patch matrix has shape {tuple(x.shape)}, expected {(kk, n)}")
        ptr = (lambda t: t.data_ptr()) if dev else (lambda t: t.ctypes.data)
        PX = (c_void_p * max(n_channels, 1))(*[ptr(x) for x in xs])
        PQ = None if same else (c_void_p * max(n_channels, 1))(*[ptr(q) for q in qs])
        self._bind_stream(dev)
        flags = 0
        if dev:
            flags |= _lib.ALL_DEVICE
            if out is None:
                out = torch.zeros((n_alph, kh, kw, C, F), dtype=torch.float64, device=W.device)
            pout = out.data_ptr()
            if not sync:
                flags |= _lib.NO_SYNC
        else:
            if out is None:
                out = np.zeros((n_alph, kh, kw, C, F), dtype=np.float64)
            pout = out.ctypes.data
        sc = _scale_args(scales, n_alph, (C, F))
        st = _lib.GpfqStats()
        args = (self._ctx, PX, PQ, n, kk, c_void_p(ptr(W)), C, F, int(c0), n_channels, flat.ctypes.data_as(POINTER(c_double)),
                K.ctypes.data_as(POINTER(c_int32)), n_alph, c_void_p(pout), flags, byref(st))
        with self._rounding(seeds, n_alph), self._penalty(l1_penalty, n_alph):
            rc = self._lib.gpfq_conv_channels(*args) if sc is None else self._lib.gpfq_conv_channels_scaled(*args, _dptr(sc))
        self._check(rc)
        self.last_stats = st.as_dict()
        return out[0] if single else out

    @staticmethod
    def _check_groups(groups, C, Cg, F):
        """A grouped kernel is (kh, kw, C / groups, F) and F is a multiple of groups."""
        groups = int(groups)
        if groups < 1 or Cg * groups != C or F % groups:
            raise ValueError(f"groups={groups} does not fit {C} input channels, a kernel with {Cg} input channels and {F} filters "
                             "(need C == W.shape[2] * groups and F % groups == 0)")
        return groups

    def conv_layer_nhwc(self, act, actq, W, alphabets, strides=(1, 1), padding="SAME", rate=(1, 1), c0=0,
                        n_channels=None, out=None, sync=True, groups=1, scales=None, seeds=None, l1_penalty=None):
        """Quantize a Conv2D kernel straight from the NHWC activations (on-device patch extraction).  With `groups` > 1, W is the
        (kh, kw, C / groups, F) kernel of a grouped Conv2D: input channel c is walked against the F / groups filters of its group
        c // (C / groups); c0 / n_channels index input channels.  The result has W's shape.  `scales` (per-channel alphabets):
        (C / groups, F) or (n_alphabets, C / groups, F), indexed like W's last two axes.  `seeds` as in `dense_layer`; the slice
        W[:, :, ci, f] draws as unit ci * F + f.  `l1_penalty` as in `dense_layer`."""
        flat, K, n_alph, als = _alph_args(alphabets)
        single = isinstance(alphabets, np.ndarray) and alphabets.ndim == 1
        W = self._f32(W, "W")
        act = self._f32(act, "act")
        same = actq is None or actq is act
        actq = act if same else self._f32(actq, "actq")
        dev = _is_torch(W)
        if _is_torch(act) != dev or _is_torch(actq) != dev:
            raise TypeError("act, actq and W must all be NumPy arrays or all be CUDA tensors")
        if not dev:
            act = np.ascontiguousarray(act)
            actq = act if same else np.ascontiguousarray(actq)
            W = np.ascontiguousarray(W)
        elif not (act.is_contiguous() and actq.is_contiguous() and W.is_contiguous()):
            raise ValueError("device tensors must be contiguous")
        kh, kw, Cg, F = (int(v) for v in W.shape)
        n_img, H, Wd, C = (int(v) for v in act.shape)
        if tuple(actq.shape) != tuple(act.shape):
            raise ValueError("activation / kernel channel mismatch")
        if groups == 1 and Cg != C:
            raise ValueError("activation / kernel channel mismatch")
        groups = self._check_groups(groups, C, Cg, F)
        n_channels = (C - c0) if n_channels is None else int(n_channels)
        rate = tuple(rate) if rate else (1, 1)
        ptr = (lambda t: t.data_ptr()) if dev else (lambda t: t.ctypes.data)
        self._bind_stream(dev)
        flags = 0
        if dev:
            flags |= _lib.ALL_DEVICE
            if out is None:
                out = torch.zeros((n_alph, kh, kw, Cg, F), dtype=torch.float64, device=W.device)
            pout = out.data_ptr()
            if not sync:
                flags |= _lib.NO_SYNC
        else:
            if out is None:
                out = np.zeros((n_alph, kh, kw, Cg, F), dtype=np.float64)
            pout = out.ctypes.data
        sc = _scale_args(scales, n_alph, (Cg, F))
        st = _lib.GpfqStats()
        args = (self._ctx, c_void_p(ptr(act)), c_void_p(ptr(actq)), n_img, H, Wd, C, kh, kw, int(strides[0]), int(strides[1]),
                int(rate[0]), int(rate[1]), 1 if str(padding).upper() == "SAME" else 0, c_void_p(ptr(W)), F, int(c0), n_channels,
                flat.ctypes.data_as(POINTER(c_double)), K.ctypes.data_as(POINTER(c_int32)), n_alph, c_void_p(pout), flags,
                byref(st))
        with self._rounding(seeds, n_alph), self._penalty(l1_penalty, n_alph):
            if sc is not None:
                rc = self._lib.gpfq_conv_layer_nhwc_scaled(*args, groups, _dptr(sc))
            else:
                rc = (self._lib.gpfq_conv_layer_nhwc_grouped(*args, groups) if groups > 1 else self._lib.gpfq_conv_layer_nhwc(*args))
        self._check(rc)
        self.last_stats = st.as_dict()
        return out[0] if single else out

    def conv_gram_nhwc(self, act, actq, kernel_size=(3, 3), strides=(1, 1), padding="SAME", rate=(1, 1), c0=0, n_channels=None,
                       sync=True):
        """Gram stage of a conv layer alone: per-channel [G1 | G2] of channels c0..c0+n_channels-1 over the given images,
        as a float64 CUDA tensor (n_channels, 2, kh*kw, kh*kw) (lower triangles + diagonals valid).  act / actq: NHWC
        NumPy arrays or CUDA tensors.  The per-rank part of an image-split multi-GPU job (`conv_layer_from_gram`).  Raises
        GpfqError for kh * kw outside CONV_SUPPORTED_KK (kernels above 128 taps)."""
        act = self._f32(act, "act")
        same = actq is None or actq is act
        actq = act if same else self._f32(actq, "actq")
        dev = _is_torch(act)
        if _is_torch(actq) != dev:
            raise TypeError("act and actq must both be NumPy arrays or both be CUDA tensors")
        if not dev:
            act = np.ascontiguousarray(act)
            actq = act if same else np.ascontiguousarray(actq)
        elif not (act.is_contiguous() and actq.is_contiguous()):
            raise ValueError("device tensors must be contiguous")
        if tuple(actq.shape) != tuple(act.shape):
            raise ValueError("act and actq must have the same shape")
        n_img, H, Wd, C = (int(v) for v in act.shape)
        kh, kw = (int(v) for v in kernel_size)
        n_channels = (C - c0) if n_channels is None else int(n_channels)
        rate = tuple(rate) if rate else (1, 1)
        ptr = (lambda t: t.data_ptr()) if dev else (lambda t: t.ctypes.data)
        gram = torch.zeros((n_channels, 2, kh * kw, kh * kw), dtype=torch.float64,
                           device=act.device if dev else torch.device("cuda", self.device))
        self._bind_stream(True)
        flags = (_lib.X_DEVICE if dev else 0) | _lib.Q_DEVICE | (_lib.NO_SYNC if dev and not sync else 0)
        rc = self._lib.gpfq_conv_gram_nhwc(self._ctx, c_void_p(ptr(act)), c_void_p(ptr(actq)), n_img, H, Wd, C, kh, kw,
                                           int(strides[0]), int(strides[1]), int(rate[0]), int(rate[1]),
                                           1 if str(padding).upper() == "SAME" else 0, int(c0), n_channels,
                                           c_void_p(gram.data_ptr()), flags)
        self._check(rc)
        self.last_stats = self.query_stats(0)
        return gram

    def conv_layer_from_gram(self, gram, W, alphabets, c0=0, n_channels=None, out=None, sync=True, groups=1, scales=None,
                             seeds=None, l1_penalty=None):
        """Walks of every filter of channels c0..c0+n_channels-1 from per-channel Gram matrices on the device
        (`conv_gram_nhwc`, summed over the ranks of an image-split job).  W: (kh, kw, C, F) NumPy array or CUDA tensor; with
        `groups` > 1 the (kh, kw, C / groups, F) kernel of a grouped Conv2D, each input channel walked against the F / groups
        filters of its group (c0 / n_channels index input channels, as in the Gram stage).  `scales`, `seeds` and `l1_penalty` as
        in `conv_layer_nhwc`."""
        flat, K, n_alph, als = _alph_args(alphabets)
        single = isinstance(alphabets, np.ndarray) and alphabets.ndim == 1
        W = self._f32(W, "W")
        wdev = _is_torch(W)
        W = W.contiguous() if wdev else np.ascontiguousarray(W)
        kh, kw, Cg, F = (int(v) for v in W.shape)
        kk = kh * kw
        C = Cg * int(groups)
        groups = self._check_groups(groups, C, Cg, F)
        n_channels = (C - c0) if n_channels is None else int(n_channels)
        if (not _is_torch(gram) or gram.dtype != torch.float64 or not gram.is_cuda or not gram.is_contiguous()
                or gram.numel() != n_channels * 2 * kk * kk):
            raise TypeError(f"gram must be a contiguous float64 CUDA tensor of {n_channels} x 2 x {kk} x {kk} entries")
        self._bind_stream(True)
        flags = _lib.X_DEVICE
        if wdev:
            flags |= _lib.W_DEVICE | _lib.Q_DEVICE
            if out is None:
                out = torch.zeros((n_alph, kh, kw, Cg, F), dtype=torch.float64, device=W.device)
            pout, pw = out.data_ptr(), W.data_ptr()
            if not sync:
                flags |= _lib.NO_SYNC
        else:
            if out is None:
                out = np.zeros((n_alph, kh, kw, Cg, F), dtype=np.float64)
            pout, pw = out.ctypes.data, W.ctypes.data
        sc = _scale_args(scales, n_alph, (Cg, F))
        st = _lib.GpfqStats()
        args = (self._ctx, c_void_p(gram.data_ptr()), kk, c_void_p(pw), C, F, int(c0), n_channels,
                flat.ctypes.data_as(POINTER(c_double)), K.ctypes.data_as(POINTER(c_int32)), n_alph, c_void_p(pout), flags, byref(st))
        with self._rounding(seeds, n_alph), self._penalty(l1_penalty, n_alph):
            if sc is not None:
                rc = self._lib.gpfq_conv_layer_from_gram_scaled(*args, groups, _dptr(sc))
            else:
                rc = (self._lib.gpfq_conv_layer_from_gram_grouped(*args, groups) if groups > 1
                      else self._lib.gpfq_conv_layer_from_gram(*args))
        self._check(rc)
        self.last_stats = st.as_dict()
        return out[0] if single else out

    def debug_slgemm(self, A, B, D=7, transposed_b=False):
        """C = A B^T through the int8-slice tcgen05 contraction of the residual-form sweep (diagnostics / tests).
        A: (M, K) float64; B: (N, K) float32, or (K, N) with `transposed_b`."""
        A = np.ascontiguousarray(A, dtype=np.float64)
        B = np.ascontiguousarray(B, dtype=np.float32)
        M, K = A.shape
        N = B.shape[1] if transposed_b else B.shape[0]
        if (B.shape[0] if transposed_b else B.shape[1]) != K:
            raise ValueError("A and B disagree on K")
        C = np.zeros((M, N), dtype=np.float64)
        self._bind_stream(False)
        self._check(self._lib.gpfq_debug_slgemm(self._ctx, c_void_p(A.ctypes.data), c_void_p(B.ctypes.data), M, N, K, int(D),
                                                1 if transposed_b else 0, c_void_p(C.ctypes.data)))
        return C

    def msq(self, W, alphabet, scales=None, seeds=None):
        """Plain nearest-level rounding of every weight (the MSQ baseline of the reference's drivers).  `scales` (per-channel
        alphabets): one scale per unit of W's last axis (a Dense neuron or a conv filter), shape (W.shape[-1],) or W.shape[-2:]
        for a conv kernel's (C, F) table; weight W[..., u] rounds to the levels fl64(scales[u] * alphabet[k]).  `seeds` (one int):
        stochastic rounding, the flat element index as unit id."""
        W = np.ascontiguousarray(W, dtype=np.float32)
        A = np.ascontiguousarray(alphabet, dtype=np.float64)
        out = np.zeros(W.shape, dtype=np.float64)
        self._bind_stream(False)
        if scales is not None:
            s = np.asarray(scales.detach().cpu().numpy() if _is_torch(scales) else scales, dtype=np.float64)
            if W.ndim < 1 or s.shape not in (W.shape[-1:], W.shape[-2:]):
                raise ValueError(f"scales: shape {s.shape}, expected {W.shape[-1:]} or {W.shape[-2:]}")
            if not np.all(np.isfinite(s)) or np.any(s < 0):
                raise ValueError("scales: every scale must be finite and >= 0")
            s = np.ascontiguousarray(s).reshape(-1)
            with self._rounding(seeds, 1):
                rc = self._lib.gpfq_msq_scaled(self._ctx, c_void_p(W.ctypes.data), W.size, A.ctypes.data_as(POINTER(c_double)),
                                               len(A), _dptr(s), s.size, c_void_p(out.ctypes.data), 0)
            self._check(rc)
            return out
        with self._rounding(seeds, 1):
            rc = self._lib.gpfq_msq(self._ctx, c_void_p(W.ctypes.data), W.size, A.ctypes.data_as(POINTER(c_double)), len(A),
                                    c_void_p(out.ctypes.data), 0)
        self._check(rc)
        return out


    def _bit_round(self, t, alphabet, seeds=None):
        """The scalar quantizer on fp64 values; `seeds` (one int): stochastic rounding, the flat index as unit id."""
        t = np.ascontiguousarray(t, dtype=np.float64)
        A = np.ascontiguousarray(alphabet, dtype=np.float64)
        out = np.zeros(t.shape, dtype=np.float64)
        self._bind_stream(False)
        with self._rounding(seeds, 1):
            rc = self._lib.gpfq_bit_round(self._ctx, c_void_p(t.ctypes.data), t.size, A.ctypes.data_as(POINTER(c_double)),
                                          len(A), c_void_p(out.ctypes.data), 0)
        self._check(rc)
        return out

    bit_round = _bit_round


_engines = {}


def get_engine(device: int = 0) -> GpfqEngine:
    """Process-wide engine per device (one context per GPU per process)."""
    if device not in _engines:
        _engines[device] = GpfqEngine(device)
    return _engines[device]
