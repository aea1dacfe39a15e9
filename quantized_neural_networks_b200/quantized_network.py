"""Host-side mirror of the reference's `scripts/quantized_network.py` API over libgpfq.

Same classes, constructor signatures, method names and attributes as the reference
(`QuantizedNeuralNetwork` quantized_network.py:331-590, `QuantizedCNN` :592-883, and the module-level
workers `_bit_round_parallel` :40, `_quantize_neuron_parallel` :91, `_quantize_filter2D_parallel_jit`
:185), so a driver script written against the reference runs unchanged.  What differs is below the
override points named in SURVEY.md section 8b:

  * activation collection stays host Python (as BASELINE.json's north_star prescribes) but hands
    NumPy matrices to CUDA instead of writing `layer{idx}_data.h5` / `channel{c}_patch_array.h5`;
  * the process-pool fan-out over neurons / filters (:549-567, :706-721) and the N0-step walks they run
    are ONE call into the C ABI (`gpfq_dense_layer`, `gpfq_conv_channels`, `gpfq_conv_layer_nhwc`).

Works with real Keras models when TensorFlow is importable and with `hostnet` models otherwise.
There is no CPU fallback for the hot path: without libgpfq.so and an sm_100 GPU the calls raise.
"""
from __future__ import annotations

import numbers
from collections.abc import Mapping
from time import time
from typing import List

import numpy as np
from numpy import abs, array, linspace, log2, median, zeros

from . import hostnet
from .engine import CONV_SUPPORTED_KK, get_engine
from .replicate import image_split_conv_gram, prefer_sample_split, replicate_leading_axis, sample_split_gram, shard_range

try:  # real Keras if present, the TF-free shim otherwise (same call surface, SURVEY.md App. D)
    from tensorflow.keras.models import Model as _KModel, clone_model as _kclone  # type: ignore
except Exception:  # pragma: no cover - TensorFlow is absent in the build image
    _KModel, _kclone = None, None


def _clone(network):
    if isinstance(network, hostnet.Sequential) or _kclone is None:
        return hostnet.clone_model(network)
    return _kclone(network)


def _partial_model(net, layers):
    if isinstance(net, hostnet.Sequential) or _KModel is None:
        return hostnet.Model(inputs=net.layers[0].input, outputs=[l.output for l in layers])
    return _KModel(inputs=net.layers[0].input, outputs=[l.output for l in layers])


# ---------------------------------------------------------------------------------------------
# module-level workers (finest-grain swap points of the reference)
# ---------------------------------------------------------------------------------------------
def _bit_round_parallel(t: float, alphabet: array, device: int = 0) -> float:
    """Nearest alphabet element, ties to the lower index (quantized_network.py:40-57), on the GPU."""
    return float(get_engine(device).bit_round(np.asarray([t], dtype=np.float64), alphabet)[0])


def _layer_arrays(data):
    """Accept what `_get_layer_data_generator` returns here: an object/dict with wX, qX (feature-major)."""
    if isinstance(data, dict):
        return data["wX"], data["qX"]
    return data.wX, data.qX


def _quantize_neuron_parallel(w: array, hf_filename, alphabet: array, device: int = 0) -> array:
    """One Dense neuron (quantized_network.py:91-121).  `hf_filename` is the in-memory layer data
    (wX, qX of shape (N0, m)) that replaces the reference's HDF5 file name."""
    wX, qX = _layer_arrays(hf_filename)
    W = np.ascontiguousarray(np.asarray(w, dtype=np.float32).reshape(-1, 1))
    Q = get_engine(device).dense_layer(wX, None if qX is wX else qX, W, np.asarray(alphabet, dtype=np.float64))
    return Q[:, 0].copy()


def _quantize_filter2D_parallel_jit(chan_filter: array, channel_idx: int, channel_hf_filename, alphabet: array,
                                    device: int = 0) -> array:
    """One (kh, kw) channel filter (quantized_network.py:185-233).  `channel_hf_filename` is the in-memory
    patch data: a dict with `wX_channel{c}` / `qX_channel{c}` of shape (kh*kw, n_patches)."""
    Xp = channel_hf_filename[f"wX_channel{channel_idx}"]
    Xqp = channel_hf_filename[f"qX_channel{channel_idx}"]
    f = np.asarray(chan_filter, dtype=np.float32)
    W = np.ascontiguousarray(f.reshape(f.size, 1))
    Q = get_engine(device).dense_layer(Xp, None if Xqp is Xp else Xqp, W, np.asarray(alphabet, dtype=np.float64))
    return Q[:, 0].reshape(f.shape)


class LayerData:
    """In-memory replacement of `layer{idx}_data.h5` (datasets wX, qX; quantized_network.py:471-500)."""

    def __init__(self, wX, qX):
        self.wX, self.qX = wX, qX
        self.same = qX is wX or np.array_equal(wX, qX)


_MASK64 = (1 << 64) - 1


def splitmix64(x: int) -> int:
    """The SplitMix64 finaliser of x + 0x9E3779B97F4A7C15 (mod 2^64): the hash of the stochastic-rounding draws (include/gpfq.h)."""
    z = (x + 0x9E3779B97F4A7C15) & _MASK64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _MASK64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _MASK64
    return z ^ (z >> 31)


def layer_seed(seed: int, layer_idx: int) -> int:
    """The stochastic-rounding seed of layer `layer_idx` of a network quantized with `seed`: every layer draws its own stream,
    and a layer's decisions do not depend on which other layers are quantized."""
    return splitmix64(splitmix64(int(seed) & _MASK64) ^ int(layer_idx))


def _check_l1_penalty(l1_penalty, alphabet):
    """The `l1_penalty` argument of the mirror classes, validated: None, a float, or a dict {layer_idx: float}."""
    if l1_penalty is None:
        return None

    def one(v, what):
        if isinstance(v, bool) or not isinstance(v, numbers.Real) or not np.isfinite(float(v)) or float(v) < 0:
            raise ValueError(f"l1_penalty{what} must be a finite number >= 0, not {v!r}")
        return float(v)

    if isinstance(l1_penalty, Mapping):
        out = {}
        for k, v in l1_penalty.items():
            if isinstance(k, bool) or not isinstance(k, numbers.Integral):
                raise ValueError(f"l1_penalty: layer index {k!r} is not an int")
            out[int(k)] = one(v, f"[{k}]")
        lams = out
    else:
        lams = one(l1_penalty, "")
    if not np.any(np.asarray(alphabet) == 0.0):
        raise ValueError(f"l1_penalty needs an alphabet with a 0 level, and linspace(-1, 1, {len(alphabet)}) has none: soft "
                         "thresholding only makes zeros with an odd number of levels K, bits = log2(2K + 1) (log2(3), log2(5), ...)")
    return lams


class QuantizedNeuralNetwork:
    def __init__(
        self,
        network,
        batch_size: int,
        get_data,
        mini_batch_size=32,
        logger=None,
        ignore_layers=[],
        bits=log2(3),
        alphabet_scalar=1,
        *,
        device: int = 0,
        method: str = "auto",
        shard=None,
        gram_split: str = "auto",
        alphabet_scope: str = "layer",
        rounding: str = "nearest",
        seed: int = 0,
        l1_penalty=None,
    ):
        """Wrapper of a Keras-style model that quantizes the weights of its Dense layers with GPFQ.

        Parameters are those of the reference (quantized_network.py:332-369); `batch_size` and
        `mini_batch_size` are accepted and unused there too (the sample count is
        `len(get_data) * get_data.batch_size`, :467).  Keyword-only extras: `device` (GPU index),
        `method` ("auto" | "stream" | "gram") and `shard=(rank, world)` to split every layer's neurons
        over the ranks of a torch.distributed job (Q blocks are all-gathered after each layer), and
        `gram_split` ("auto" | "samples" | "replicate"): how a multi-GPU job feeds a Dense layer -- "samples" contracts
        m / world samples per rank and all-reduces the Gram matrices, "replicate" all-gathers the inputs; "auto" picks
        by bytes moved (`replicate.prefer_sample_split`).  `alphabet_scope` ("layer" | "channel"): "layer" (the reference)
        quantizes every layer against `alphabet_scalar * median(|W|) * linspace(-1, 1, K)`; "channel" gives every output
        channel its own radius `alphabet_scalar * median(|w_u|)` (`_unit_scales`), as per-channel weight scales do.
        `rounding` ("nearest" | "stochastic"): "nearest" (the reference) rounds every greedy step to the nearest level;
        "stochastic" is SPFQ, unbiased stochastic rounding between the two bracketing levels, reproducible from `seed` (layer
        `layer_idx` draws with `layer_seed(seed, layer_idx)`, whatever the device count, shards or conv path).
        `l1_penalty` (sparse GPFQ): None (the reference) or a finite lambda >= 0 for every quantized layer, or a mapping
        {layer_idx: lambda} (layers not in it walk without the penalty).  Every greedy step's value is then soft-thresholded by
        lambda / nrm^2 before it is quantized (include/gpfq.h), so the layer is pruned and quantized in one pass; the alphabet
        needs a 0 level (odd K: bits = log2(2K + 1)).
        """
        self.get_data = get_data
        self.trained_net = network
        self.quantized_net = _clone(network)
        self.quantized_net.set_weights(network.get_weights())
        self.alphabet_scalar = alphabet_scalar
        self.layer_dims = {
            layer_idx: layer.get_weights()[0].shape
            for layer_idx, layer in enumerate(network.layers)
            if layer.__class__.__name__ == "Dense"
        }
        self.bits = bits
        self.alphabet = linspace(-1, 1, num=int(round(2 ** (bits))))
        self.logger = logger
        self.ignore_layers = ignore_layers
        self._init_device(device, method, shard, gram_split, alphabet_scope, rounding, seed, l1_penalty)

    def _init_device(self, device, method, shard, gram_split="auto", alphabet_scope="layer", rounding="nearest", seed=0,
                     l1_penalty=None):
        if int(round(2 ** self.bits)) > 64:   # GPFQ_MAX_K of include/gpfq.h: the kernels keep an alphabet in shared memory
            raise ValueError(f"bits={self.bits}: the CUDA path supports alphabets of up to 64 levels (bits <= 6); the reference "
                             "accepts any `bits`, see INTEGRATION.md")
        if gram_split not in ("auto", "samples", "replicate"):
            raise ValueError(f"gram_split must be 'auto', 'samples' or 'replicate', not {gram_split!r}")
        if alphabet_scope not in ("layer", "channel"):
            raise ValueError(f"alphabet_scope must be 'layer' or 'channel', not {alphabet_scope!r}")
        self.alphabet_scope = alphabet_scope
        if rounding not in ("nearest", "stochastic"):
            raise ValueError(f"rounding must be 'nearest' or 'stochastic', not {rounding!r}")
        if isinstance(seed, bool) or not isinstance(seed, numbers.Integral) or not 0 <= int(seed) < 1 << 64:
            raise ValueError(f"seed must be an int in [0, 2^64), not {seed!r}")
        self.rounding, self.seed = rounding, int(seed)
        self.l1_penalty = _check_l1_penalty(l1_penalty, self.alphabet)
        self.device, self.method, self.gram_split = device, method, gram_split
        self.shard = tuple(shard) if shard else (0, 1)
        self.layer_stats = {}

    @property
    def engine(self):
        return get_engine(self.device)

    def _log(self, msg: str):
        if self.logger:
            self.logger.info(msg)
        else:
            print(msg)

    # -- host-side collection (stays Python, quantized_network.py:408-502) ---------------------
    def _get_layer_data_generator(self, layer_idx: int, transpose=False):
        """Inputs of layer `layer_idx` in the analog and the (partially) quantized network.

        Returns a `LayerData` holding float32 `wX`, `qX` of shape (num_images, *layer_input_shape), or its
        reverse when `transpose` (feature-major, what the Dense walk wants).  Rows are written exactly as
        the reference does, including its offset arithmetic for a short final batch (SURVEY.md App. E 2).
        """
        layer = self.trained_net.layers[layer_idx]
        if layer_idx == 0:
            analog_model = quant_model = None
            n_inbound = 1
        else:
            a_in = self.trained_net.layers[layer_idx].inbound_nodes[0].inbound_layers
            q_in = self.quantized_net.layers[layer_idx].inbound_nodes[0].inbound_layers
            a_in = a_in if isinstance(a_in, (list, tuple)) else [a_in]
            q_in = q_in if isinstance(q_in, (list, tuple)) else [q_in]
            assert len(a_in) == len(q_in)
            n_inbound = len(a_in)
            analog_model = _partial_model(self.trained_net, a_in)
            quant_model = _partial_model(self.quantized_net, q_in)
        in_shape = layer.input_shape
        data_shape = tuple(in_shape[1:]) if in_shape[0] is None else tuple(in_shape)
        num_images = len(self.get_data) * self.get_data.batch_size
        shape = (n_inbound * num_images, *data_shape)
        if transpose:
            shape = shape[::-1]
        wX_all = np.zeros(shape, dtype=np.float32)
        qX_all = wX_all if layer_idx == 0 else np.zeros(shape, dtype=np.float32)
        for batch_idx in range(len(self.get_data)):
            mini_batch = self.get_data[batch_idx][0]
            if layer_idx == 0:
                wX = qX = np.asarray(mini_batch, dtype=np.float32)
            else:
                wX = np.asarray(analog_model.predict_on_batch(mini_batch))
                qX = np.asarray(quant_model.predict_on_batch(mini_batch))
            b = wX.shape[0]
            if transpose:
                wX_all[..., batch_idx * b:(batch_idx + 1) * b] = wX.T
                if qX_all is not wX_all:
                    qX_all[..., batch_idx * b:(batch_idx + 1) * b] = qX.T
            else:
                wX_all[batch_idx * b:(batch_idx + 1) * b] = wX
                if qX_all is not wX_all:
                    qX_all[batch_idx * b:(batch_idx + 1) * b] = qX
        return LayerData(wX_all, qX_all)

    def _update_weights(self, layer_idx: int, Q: array):
        """Install Q in the quantized network, bias carried over unchanged (quantized_network.py:504-521)."""
        if self.trained_net.layers[layer_idx].use_bias:
            bias = self.trained_net.layers[layer_idx].get_weights()[1]
            self.quantized_net.layers[layer_idx].set_weights([Q, bias])
        else:
            self.quantized_net.layers[layer_idx].set_weights([Q])

    def _layer_alphabet(self, W):
        """`rad = alphabet_scalar * median(|W|)`; `rad * alphabet` (quantized_network.py:544-545, :831-832)."""
        rad = self.alphabet_scalar * median(abs(W.flatten()))
        return rad * self.alphabet

    def _unit_scales(self, W, kind="Dense"):
        """Per-output-channel radii `alphabet_scalar * median(|w_u|)`, the expression (and dtype) of `_layer_alphabet` applied to
        each output channel: a Dense neuron (column j: shape (N1,)), a Conv2D filter f over W[..., f] (broadcast over the kernel's
        input channels: (Cw, F)), a DepthwiseConv2D output channel (c, d) over W[:, :, c, d] (shape (C, d)).  Unit u then walks
        with the levels fl64(rad_u * linspace(-1, 1, K)), exactly `rad_u * self.alphabet`."""
        A = abs(W)
        if kind == "Dense":
            return np.asarray(self.alphabet_scalar * median(A, axis=0), dtype=np.float64)
        if kind == "DepthwiseConv2D":
            return np.asarray(self.alphabet_scalar * median(A, axis=(0, 1)), dtype=np.float64)
        rad = np.asarray(self.alphabet_scalar * median(A, axis=(0, 1, 2)), dtype=np.float64)
        return np.ascontiguousarray(np.broadcast_to(rad, W.shape[2:]))

    def _levels(self, W, kind="Dense"):
        """(alphabet, scales) of a layer: the layer alphabet and None, or the base alphabet and the per-channel radii."""
        if self.alphabet_scope == "channel":
            return np.asarray(self.alphabet, dtype=np.float64), self._unit_scales(W, kind)
        return np.asarray(self._layer_alphabet(W), dtype=np.float64), None

    def _seeds(self, layer_idx):
        """Engine keyword of layer `layer_idx`: nothing for nearest rounding (the call keeps its signature), else its seed."""
        return {"seeds": layer_seed(self.seed, layer_idx)} if self.rounding == "stochastic" else {}

    def _penalty(self, layer_idx):
        """Engine keyword of layer `layer_idx`: nothing without a penalty (the call keeps its signature), else its lambda."""
        lam = self._layer_l1(layer_idx)
        return {} if lam is None else {"l1_penalty": lam}

    def _layer_l1(self, layer_idx):
        """The L1 penalty of layer `layer_idx`, or None."""
        if isinstance(self.l1_penalty, dict):
            return self.l1_penalty.get(layer_idx)
        return self.l1_penalty

    def _nccl_job(self):
        """True when this object is one rank of a torch.distributed job on GPUs (NCCL): layer inputs are then replicated
        through `replicate_leading_axis` (1 / world of the bytes over each rank's host link + one NVLink all-gather)."""
        if self.shard[1] == 1:
            return False
        try:
            import torch.distributed as dist
            return dist.is_available() and dist.is_initialized() and dist.get_backend() == "nccl"
        except Exception:  # pragma: no cover
            return False

    def _sample_split(self, N0, m):
        """Whether a Dense layer of this multi-GPU job runs its Gram stage split over samples (+ all-reduce)."""
        if self.gram_split == "auto":
            return self.method in ("auto", "gram") and prefer_sample_split(N0, m, self.shard[1])
        return self.gram_split == "samples"

    def _replicated(self, *arrays):
        """Device copies of host arrays every rank holds; `None` entries pass through."""
        import torch
        dev = torch.device("cuda", self.device)
        rank, world = self.shard
        return [None if a is None else replicate_leading_axis(a, rank, world, dev) for a in arrays]

    def _gather_columns(self, Q, lo, hi, axis):
        """All-gather the shard's block of Q over the job (multi-GPU); identity for a single rank."""
        rank, world = self.shard
        if world == 1:
            return Q
        import torch
        import torch.distributed as dist
        n = Q.shape[axis]
        width = -(-n // world)
        blk = np.zeros([width if a == axis else s for a, s in enumerate(Q.shape)])
        sl = [slice(None)] * Q.ndim
        sl[axis] = slice(lo, hi)
        dst = [slice(None)] * Q.ndim
        dst[axis] = slice(0, hi - lo)
        blk[tuple(dst)] = Q[tuple(sl)]
        t = torch.from_numpy(np.ascontiguousarray(blk))
        use_cuda = dist.get_backend() == "nccl"
        if use_cuda:
            t = t.cuda(self.device)
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        out = np.zeros_like(Q)
        for r, p in enumerate(parts):
            rlo, rhi = shard_range(n, r, world)
            sl[axis] = slice(rlo, rhi)
            dst[axis] = slice(0, rhi - rlo)
            out[tuple(sl)] = p.cpu().numpy()[tuple(dst)]
        return out

    def _quantize_layer_parallel(self, layer_idx: int):
        """Quantizes a Dense layer (quantized_network.py:523-574): one C-ABI call instead of a process pool."""
        W = self.trained_net.layers[layer_idx].get_weights()[0]
        N_ell, N_ell_plus_1 = W.shape
        self._log("\tFeeding input data through hidden layers...")
        tic = time()
        data = self._get_layer_data_generator(layer_idx, transpose=True)
        self._log(f"\tdone. {time()-tic:2f} seconds.")

        layer_alphabet, scales = self._levels(W)
        scaled = {"scales": scales} if scales is not None else {}   # the per-layer call keeps its signature
        scaled.update(self._seeds(layer_idx))
        scaled.update(self._penalty(layer_idx))

        self._log("\tQuantizing neurons (on the GPU)...")
        tic = time()
        lo, hi = shard_range(N_ell_plus_1, *self.shard)
        try:
            if self._nccl_job() and self._sample_split(N_ell, data.wX.shape[1]):
                import torch
                dev = torch.device("cuda", self.device)
                G1, G2 = sample_split_gram(self.engine, data.wX, None if data.same else data.qX, *self.shard, device=dev)
                Q = self.engine.dense_layer_from_gram(G1, G2, np.ascontiguousarray(W),
                                                      np.asarray(layer_alphabet, dtype=np.float64), j0=lo, j1=hi, **scaled)
            elif self._nccl_job():
                import torch
                Xd, Xqd = self._replicated(data.wX, None if data.same else data.qX)
                Wd = torch.from_numpy(np.ascontiguousarray(W)).to(Xd.device)
                Q = self.engine.dense_layer(Xd, Xqd, Wd, np.asarray(layer_alphabet, dtype=np.float64), j0=lo, j1=hi,
                                            method=self.method, **scaled).cpu().numpy()
            else:
                Q = self.engine.dense_layer(data.wX, None if data.same else data.qX, np.ascontiguousarray(W),
                                            np.asarray(layer_alphabet, dtype=np.float64), j0=lo, j1=hi, method=self.method,
                                            **scaled)
        except Exception as exc:
            self._log(f"\t\tNeurons {lo}:{hi} generated an exception: {exc}")
            raise exc
        self.layer_stats[layer_idx] = dict(self.engine.last_stats)
        Q = self._gather_columns(Q, lo, hi, axis=1)
        self._log(f"\t\t{N_ell_plus_1} neurons x {N_ell} weights quantized successfully.")
        self._update_weights(layer_idx, Q)
        self._log(f"\tdone. {time()-tic:.2f} seconds.")

    def quantize_network(self):
        """Quantizes all Dense layers that are not specified by the list of ignored layers (sequentially, :576-590)."""
        num_layers = len(self.trained_net.layers)
        for layer_idx, layer in enumerate(self.trained_net.layers):
            if layer.__class__.__name__ == "Dense" and layer_idx not in self.ignore_layers:
                tic = time()
                self._log(f"Quantizing layer {layer_idx} (in parallel) of {num_layers}...")
                self._quantize_layer_parallel(layer_idx)
                self._log(f"Layer {layer_idx} of {num_layers} quantized successfully in {time() - tic:.2f} seconds.")


class QuantizedCNN(QuantizedNeuralNetwork):
    def __init__(
        self,
        network,
        batch_size: int,
        get_data,
        mini_batch_size=32,
        logger=None,
        bits=log2(3),
        alphabet_scalar=1,
        patch_mini_batch_size=5000,
        is_quantize_conv2d=True,
        *,
        device: int = 0,
        method: str = "auto",
        shard=None,
        conv_path: str = "nhwc",
        gram_split: str = "auto",
        alphabet_scope: str = "layer",
        rounding: str = "nearest",
        seed: int = 0,
        l1_penalty=None,
    ):
        """Dense + Conv2D / DepthwiseConv2D quantization (quantized_network.py:594-650).  Like the reference this
        constructor does not take `ignore_layers`.  `conv_path="nhwc"` hands the layer's activation tensors to
        CUDA (patches are extracted on the device); `"patches"` builds the per-channel patch matrices on the host
        exactly as `_build_patch_array` does and hands those over.  `alphabet_scope`, `rounding`, `seed` and `l1_penalty` as
        in `QuantizedNeuralNetwork`."""
        self.get_data = get_data
        self.trained_net = network
        self.quantized_net = _clone(network)
        self.quantized_net.set_weights(network.get_weights())
        self.patch_mini_batch_size = patch_mini_batch_size
        self.is_quantize_conv2d = is_quantize_conv2d
        self.alphabet_scalar = alphabet_scalar
        self.bits = bits
        self.alphabet = linspace(-1, 1, num=int(round(2 ** (bits))))
        self.logger = logger
        self.ignore_layers = []
        self.conv_path = conv_path
        self._init_device(device, method, shard, gram_split, alphabet_scope, rounding, seed, l1_penalty)

    def _build_patch_array(self, channel_idx: int, kernel_size: tuple, strides: tuple, padding: str, rate: tuple,
                           data, mini_batch_size: int):
        """Patch matrices of one channel, (kh*kw, n_patches) float32 each (quantized_network.py:729-809), in memory."""
        rates = [1, *rate, 1] if rate else [1, 1, 1, 1]
        out = []
        for arr in ((data.wX,) if data.same else (data.wX, data.qX)):
            cols = []
            for s in range(0, arr.shape[0], mini_batch_size):
                ch = arr[s:s + mini_batch_size, ..., channel_idx]
                seg = hostnet.extract_patches(ch.reshape(*ch.shape, 1), [1, *kernel_size, 1], [1, *strides, 1], rates, padding)
                cols.append(seg.reshape(-1, seg.shape[-1]).T)
            out.append(np.ascontiguousarray(np.concatenate(cols, axis=1)))
        wXp = out[0]
        qXp = wXp if data.same else out[1]
        return {f"wX_channel{channel_idx}": wXp, f"qX_channel{channel_idx}": qXp}

    def _quantize_channel_parallel_jit(self, channel_idx: int, channel_filters: array, hidden_activations,
                                       strides: tuple, padding: str, rate: tuple, alphabet: array,
                                       patch_mini_batch_size=5000, scales=None, stochastic=None, l1_penalty=None) -> array:
        """All filters of one input channel (quantized_network.py:652-727): host patches + one C-ABI call.  `stochastic`
        (stochastic rounding): (kernel, ci, f0, seed, scales) -- the whole (kh, kw, Cw, F) kernel, the channel's slice ci and its
        first filter f0, so that the slice draws with its global unit ids ci * F + f; the call walks all F filters of slice ci and
        the Fg of `channel_filters` are kept.  `l1_penalty`: the layer's lambda, or None."""
        pen = {} if l1_penalty is None else {"l1_penalty": l1_penalty}
        filter_shape = channel_filters.shape[0:2]
        patches = self._build_patch_array(channel_idx, filter_shape, strides, padding, rate, hidden_activations,
                                          patch_mini_batch_size)
        Xp, Xqp = patches[f"wX_channel{channel_idx}"], patches[f"qX_channel{channel_idx}"]
        Wc = np.ascontiguousarray(channel_filters.reshape(*channel_filters.shape[:2], 1, channel_filters.shape[-1]),
                                  dtype=np.float32)
        try:
            if stochastic is not None:
                Wk, ci, f0, seed, sk = stochastic
                Qk = self.engine.conv_channels([Xp], None if Xqp is Xp else [Xqp], np.ascontiguousarray(Wk, dtype=np.float32),
                                               np.asarray(alphabet, dtype=np.float64), c0=ci, n_channels=1, seeds=seed,
                                               **({} if sk is None else {"scales": sk}), **pen)
                return Qk[:, :, ci, f0:f0 + channel_filters.shape[-1]]
            scaled = {} if scales is None else {"scales": np.reshape(scales, (1, -1))}
            Qc = self.engine.conv_channels([Xp], None if Xqp is Xp else [Xqp], Wc, np.asarray(alphabet, dtype=np.float64), **scaled,
                                           **pen)
        except Exception as exc:
            self._log(f"\t\t\tChannel {channel_idx} generated an exception: {exc}")
            raise Exception
        return Qc[:, :, 0, :]

    def _quantize_dense_layer(self, layer_idx: int):
        super()._quantize_layer_parallel(layer_idx)

    def _quantize_conv2D_layer_parallel_jit(self, layer_idx: int):
        """One Conv2D / DepthwiseConv2D layer (quantized_network.py:815-867); channels sharded over ranks."""
        self._log("\tFeeding input data through hidden layers...")
        tic = time()
        data = self._get_layer_data_generator(layer_idx)
        self._log(f"\tdone. {time()-tic:.2f} seconds.")
        layer = self.trained_net.layers[layer_idx]
        rate = getattr(layer, "dilation_rate", None)
        W = layer.get_weights()[0]
        alphabet, scales = self._levels(W, layer.__class__.__name__)
        scaled = {"scales": scales} if scales is not None else {}
        scaled.update(self._seeds(layer_idx))
        scaled.update(self._penalty(layer_idx))
        # a grouped Conv2D has a (kh, kw, C / groups, F) kernel: input channel c meets only the Fg filters of its group c // Cg,
        # so ranks take whole groups and gather their filters (groups == 1: channels, all filters)
        groups = int(getattr(layer, "groups", 1)) if layer.__class__.__name__ == "Conv2D" else 1
        grouped = {"groups": groups} if groups > 1 else {}   # the ungrouped call keeps its signature
        Cg, Fg = W.shape[-2], W.shape[-1] // groups
        num_channels = Cg * groups
        unit = Cg if groups > 1 else 1
        lo, hi = (u * unit for u in shard_range(num_channels // unit, *self.shard))
        tic = time()
        if self.conv_path == "nhwc":
            try:
                if self._nccl_job() and self.gram_split != "replicate" and W.shape[0] * W.shape[1] in CONV_SUPPORTED_KK:
                    # image split: every rank contracts n_img / world images of ALL channels, one tiny all-reduce sums the
                    # per-channel Grams, then every rank walks every channel (cheap: kk steps per filter) -- no Q gather.
                    # Kernels above 128 taps (13 x 11, ...) have no Gram-only path and take the channel shards below.
                    gram = image_split_conv_gram(self.engine, data.wX, None if data.same else data.qX, W.shape[:2],
                                                 layer.strides, layer.padding.upper(), rate, *self.shard)
                    self.layer_stats[layer_idx] = dict(self.engine.last_stats)
                    Q = self.engine.conv_layer_from_gram(gram, np.ascontiguousarray(W), np.asarray(alphabet, dtype=np.float64),
                                                         **grouped, **scaled)
                    lo, hi = 0, num_channels
                elif self._nccl_job():
                    import torch
                    Ad, Aqd = self._replicated(data.wX, None if data.same else data.qX)
                    Wd = torch.from_numpy(np.ascontiguousarray(W)).to(Ad.device)
                    Q = self.engine.conv_layer_nhwc(Ad, Aqd, Wd, np.asarray(alphabet, dtype=np.float64), strides=layer.strides,
                                                    padding=layer.padding.upper(), rate=rate, c0=lo,
                                                    n_channels=hi - lo, **grouped, **scaled).cpu().numpy()
                else:
                    Q = self.engine.conv_layer_nhwc(data.wX, None if data.same else data.qX, np.ascontiguousarray(W),
                                                    np.asarray(alphabet, dtype=np.float64), strides=layer.strides,
                                                    padding=layer.padding.upper(), rate=rate, c0=lo, n_channels=hi - lo,
                                                    **grouped, **scaled)
            except Exception as exc:
                self._log(f"\t\tChannels {lo}:{hi} generated an exception: {exc}")
                raise exc
            self.layer_stats.setdefault(layer_idx, dict(self.engine.last_stats))
        else:
            Q = zeros(W.shape)
            for channel_idx in range(lo, hi):
                ci, f0 = channel_idx % Cg, (channel_idx // Cg) * Fg   # the channel's kernel slice and its group's filters
                stoch = (W, ci, f0, scaled["seeds"], scales) if "seeds" in scaled else None
                Q[:, :, ci, f0:f0 + Fg] = self._quantize_channel_parallel_jit(
                    channel_idx, W[:, :, ci, f0:f0 + Fg], data, strides=layer.strides, padding=layer.padding.upper(),
                    rate=rate, alphabet=alphabet, patch_mini_batch_size=self.patch_mini_batch_size,
                    scales=None if scales is None else scales[ci, f0:f0 + Fg], stochastic=stoch,
                    l1_penalty=scaled.get("l1_penalty"))
        if (lo, hi) != (0, num_channels) and groups > 1:
            # this rank wrote the filters of groups lo / Cg .. hi / Cg: gather along the group axis of (kh, kw, Cg, groups, Fg)
            Q = self._gather_columns(Q.reshape(*Q.shape[:3], groups, Fg), lo // Cg, hi // Cg, axis=3).reshape(W.shape)
        elif (lo, hi) != (0, num_channels):
            Q = self._gather_columns(Q, lo, hi, axis=2)
        self._log(f"\t\t{num_channels} channels x {W.shape[-1]} filters quantized in {time()-tic:.2f} seconds.")
        self._update_weights(layer_idx, Q)

    def quantize_network(self):
        """Dense layers through the parent's path, Conv2D / DepthwiseConv2D when `is_quantize_conv2d` (:869-883)."""
        num_layers = len(self.trained_net.layers)
        for layer_idx, layer in enumerate(self.trained_net.layers):
            if layer.__class__.__name__ == "Dense":
                self._log(f"Quantizing (Dense) layer {layer_idx} of {num_layers}...")
                tic = time()
                self._quantize_dense_layer(layer_idx)
                self._log(f"done. {time() - tic:.2f} seconds.")
            if layer.__class__.__name__ in {"Conv2D", "DepthwiseConv2D"} and self.is_quantize_conv2d:
                self._log(f"Quantizing ({layer.__class__.__name__}) layer {layer_idx} of {num_layers}...")
                tic = time()
                self._quantize_conv2D_layer_parallel_jit(layer_idx)
                self._log(f"done. {time() - tic:.2f} seconds.")


__all__: List[str] = ["QuantizedNeuralNetwork", "QuantizedCNN", "LayerData", "shard_range", "layer_seed", "splitmix64",
                      "_bit_round_parallel",
                      "_quantize_neuron_parallel", "_quantize_filter2D_parallel_jit"]
