"""Grid runner: the (bits x alphabet_scalar) cross-validation of the reference's drivers as a batched workload.

The reference walks the grid one `QuantizedCNN(...).quantize_network()` at a time (`quantize_pretrained_cnn.py:32-48, :143-160`;
20 points for the CIFAR10 CNN), recomputing the analog activations and -- at the first quantized layer, where the quantized twin
still equals the analog net -- the very same Gram matrices for every point.  Here the grid points advance through the layers
in lock-step (BASELINE.json configs[4], SURVEY.md 8f rank 3):

  * the analog inputs `wX` of a layer are collected ONCE and stay on the GPU for all grid points;
  * grid points whose quantized inputs are identical (always the case at the first quantized layer: `qX == wX`) go down in
    ONE C-ABI call with `n_alphabets` alphabets (one Gram stage, one walk per alphabet);
  * deeper layers have one `qX` per grid point (the twins differ): one call each, `wX` and `W` shared on the device.

Every grid point ends with exactly the weights its own `QuantizedCNN(bits, alphabet_scalar).quantize_network()` run produces
(`tests/test_gpu_network.py::test_grid_runner_matches_point_by_point_runs`).  `msq_networks()` builds the MSQ baselines of
`quantize_pretrained_cnn.py:97-117` with the same per-layer alphabets; `metrics()` / `to_csv()` reproduce the CSV schema of
`:124-138`.  Level-index storage of a quantized kernel (int8 indices + radius, SURVEY.md 8f rank 4): `pack_levels`.
"""
from __future__ import annotations

from itertools import product
from time import time

import numpy as np
from numpy import abs, linspace, median

from .quantized_network import QuantizedCNN, layer_seed

LAYER_KINDS = ("Dense", "Conv2D", "DepthwiseConv2D")


def _unit_levels(alphabet, scales, shape):
    """Levels per entry of a kernel of `shape`: the alphabet itself, or with per-unit `scales` (shaped like the kernel's trailing
    axes: (N1,) for a Dense kernel, (C, F) for a conv kernel) the per-channel levels fl64(scales[u] * alphabet[k])."""
    A = np.asarray(alphabet, dtype=np.float64)
    if scales is None:
        return A
    s = np.asarray(scales, dtype=np.float64)
    if s.ndim > len(shape) or s.shape != tuple(shape[len(shape) - s.ndim:]):
        raise ValueError(f"scales of shape {s.shape} do not match the trailing axes of a kernel of shape {tuple(shape)}")
    return s[..., None] * A


def pack_levels(Q: np.ndarray, alphabet: np.ndarray, scales=None):
    """Quantized kernel -> (int8 level indices, alphabet).  Index -1 marks the literal 0.0 a dead direction produces
    (quantized_network.py:83-84), which need not be a level of an even-sized alphabet.  With per-channel alphabets, `alphabet` is
    the base alphabet and `scales` the per-unit scales (see `_unit_levels`); the indices then refer to each unit's own levels."""
    L = _unit_levels(alphabet, scales, Q.shape)
    idx = np.abs(Q[..., None] - L).argmin(-1).astype(np.int8)
    exact = np.take_along_axis(np.broadcast_to(L, Q.shape + L.shape[-1:]), idx[..., None].astype(np.int64), -1)[..., 0] == Q
    if not np.all(exact | (Q == 0.0)):
        raise ValueError("Q holds values that are neither alphabet levels nor 0.0")
    idx[~exact] = -1
    return idx, np.asarray(alphabet, dtype=np.float64)


def unpack_levels(idx: np.ndarray, alphabet: np.ndarray, scales=None) -> np.ndarray:
    L = np.broadcast_to(_unit_levels(alphabet, scales, idx.shape), idx.shape + (np.asarray(alphabet).shape[-1],))
    vals = np.take_along_axis(L, np.maximum(idx, 0)[..., None].astype(np.int64), -1)[..., 0]
    return np.where(idx < 0, 0.0, vals)


class QuantizedCNNGrid:
    """All (bits, alphabet_scalar) grid points of one network, quantized layer by layer in lock-step."""

    def __init__(self, network, batch_size, get_data, bits_list, alphabet_scalars, logger=None, is_quantize_conv2d=True,
                 device: int = 0, data_set: str = "synthetic", q_train_size=None, *, alphabet_scope: str = "layer",
                 rounding: str = "nearest", seed: int = 0, l1_penalty=None):
        """`alphabet_scope` ("layer" | "channel") as in `QuantizedCNN`: with "channel" every grid point quantizes each output
        channel against its own radius, and `msq_networks()` rounds with the same per-channel levels.  `rounding` as in
        `QuantizedCNN`; with "stochastic", grid point g (in the order of `self.grid`) is the run of `QuantizedCNN(..., seed=seed + g)`,
        and `msq_networks()` rounds stochastically with the same layer seeds.  `l1_penalty` as in `QuantizedCNN`, the same for every
        grid point (each lock-step call passes one lambda per batched alphabet; the MSQ baselines have no penalty)."""
        self.grid = list(product(bits_list, alphabet_scalars))          # the order of itertools.product in the driver
        self.points = [QuantizedCNN(network, batch_size, get_data, logger=logger, bits=b, alphabet_scalar=c,
                                    is_quantize_conv2d=is_quantize_conv2d, device=device, alphabet_scope=alphabet_scope,
                                    rounding=rounding, seed=(int(seed) + g) % (1 << 64) if rounding == "stochastic" else seed,
                                    l1_penalty=l1_penalty)
                       for g, (b, c) in enumerate(self.grid)]
        self.trained_net, self.logger, self.device = network, logger, device
        self.is_quantize_conv2d = is_quantize_conv2d
        self.data_set = data_set
        self.q_train_size = q_train_size if q_train_size is not None else len(get_data) * get_data.batch_size
        self.quantization_time = None
        self.calls = []          # (layer_idx, number of grid points served by the call): what was batched

    @property
    def quantized_nets(self):
        return [p.quantized_net for p in self.points]

    def _log(self, msg):
        (self.logger.info if self.logger else print)(msg)

    def _groups(self, qXs, wX):
        """Grid points with identical quantized inputs share a call.  Returns [(qX or None when it equals wX, [point ids])]."""
        groups = []
        for g, q in enumerate(qXs):
            for entry in groups:
                ref = wX if entry[0] is None else entry[0]
                if q is ref or (q.shape == ref.shape and np.array_equal(q, ref)):
                    entry[1].append(g)
                    break
            else:
                groups.append([None if (q is wX or np.array_equal(q, wX)) else q, [g]])
        return groups

    def quantize_network(self):
        import torch
        eng = self.points[0].engine
        dev = torch.device("cuda", self.device)
        tic_all = time()
        for layer_idx, layer in enumerate(self.trained_net.layers):
            kind = layer.__class__.__name__
            if kind not in LAYER_KINDS or (kind != "Dense" and not self.is_quantize_conv2d):
                continue
            dense = kind == "Dense"
            tic = time()
            W = layer.get_weights()[0]
            levels = [p._levels(W, kind) for p in self.points]        # (alphabet, per-channel scales or None) per grid point
            datas = [p._get_layer_data_generator(layer_idx, transpose=True) if dense else p._get_layer_data_generator(layer_idx)
                     for p in self.points]
            wX = datas[0].wX                                      # the analog inputs do not depend on the grid point
            Xd = torch.from_numpy(np.ascontiguousarray(wX)).to(dev)
            Wd = torch.from_numpy(np.ascontiguousarray(W)).to(dev)
            Qs = [None] * len(self.points)
            for qX, members in self._groups([d.wX if d.same else d.qX for d in datas], wX):
                Xqd = None if qX is None else torch.from_numpy(np.ascontiguousarray(qX)).to(dev)
                A = [levels[g][0] for g in members]
                scaled = {} if levels[0][1] is None else {"scales": np.stack([levels[g][1] for g in members])}
                if self.points[0].rounding == "stochastic":
                    scaled["seeds"] = [layer_seed(self.points[g].seed, layer_idx) for g in members]
                if self.points[0]._layer_l1(layer_idx) is not None:
                    scaled["l1_penalty"] = [self.points[g]._layer_l1(layer_idx) for g in members]
                if dense:
                    Q = eng.dense_layer(Xd, Xqd, Wd, A, **scaled)
                else:
                    rate = getattr(layer, "dilation_rate", None)
                    groups = int(getattr(layer, "groups", 1)) if kind == "Conv2D" else 1
                    Q = eng.conv_layer_nhwc(Xd, Xqd, Wd, A, strides=layer.strides, padding=layer.padding.upper(), rate=rate,
                                            **({"groups": groups} if groups > 1 else {}), **scaled)
                Q = Q.cpu().numpy()
                for a, g in enumerate(members):
                    Qs[g] = Q[a]
                self.calls.append((layer_idx, len(members)))
                del Xqd
            for p, Q in zip(self.points, Qs):
                p._update_weights(layer_idx, Q)
            self._log(f"Layer {layer_idx} ({kind}) quantized for {len(self.points)} grid points in {time() - tic:.2f} seconds "
                      f"({sum(1 for c in self.calls if c[0] == layer_idx)} call(s)).")
            del Xd, Wd
        self.quantization_time = time() - tic_all
        return self

    def msq_networks(self):
        """MSQ baselines (quantize_pretrained_cnn.py:97-117): every Dense / Conv2D kernel rounded to the layer alphabet of the
        corresponding grid point (per-channel levels with `alphabet_scope="channel"`), biases and all other layers untouched."""
        from .quantized_network import _clone
        eng = self.points[0].engine
        nets = []
        for p in self.points:
            net = _clone(self.trained_net)
            net.set_weights(self.trained_net.get_weights())
            for layer_idx, layer in enumerate(self.trained_net.layers):
                if layer.__class__.__name__ in ("Dense", "Conv2D"):
                    ws = layer.get_weights()
                    A, scales = p._levels(ws[0], layer.__class__.__name__)
                    Q = eng.msq(ws[0], A, **({} if scales is None else {"scales": scales}), **p._seeds(layer_idx))
                    net.layers[layer_idx].set_weights([Q] + list(ws[1:]))
            nets.append(net)
        return nets

    @staticmethod
    def _accuracy(net, x, y):
        pred = np.asarray(net.predict(x)).argmax(-1)
        y = np.asarray(y)
        return float(np.mean(pred == (y.argmax(-1) if y.ndim > 1 else y)))

    def metrics(self, x_test, y_test):
        """One row per grid point with the columns of the reference's CSV (quantize_pretrained_cnn.py:124-138)."""
        analog = self._accuracy(self.trained_net, x_test, y_test)
        rows = []
        for (bits, c), p, msq in zip(self.grid, self.points, self.msq_networks()):
            rows.append({"data_set": self.data_set, "serialized_model": f"quantized_{self.data_set}_scaler{c}_{bits}bits",
                         "q_train_size": self.q_train_size, "ignore_layers": [], "bits": bits, "alphabet_scalar": c,
                         "analog_test_acc": analog, "sd_test_acc": self._accuracy(p.quantized_net, x_test, y_test),
                         "msq_test_acc": self._accuracy(msq, x_test, y_test),
                         "quantization_time": None if self.quantization_time is None else self.quantization_time / len(self.grid)})
        return rows

    def to_csv(self, path, x_test, y_test):
        import pandas as pd
        df = pd.DataFrame(self.metrics(x_test, y_test))
        df.to_csv(path)
        return df


def top_k_accuracy(pred: np.ndarray, labels: np.ndarray, k: int = 1) -> float:
    """Top-k accuracy of class scores `pred` (n, classes) against integer or one-hot labels -- the top-1 / top-5 figures
    of quantize_pretrained_imagenet.py:203-226."""
    labels = np.asarray(labels)
    lab = labels.argmax(-1) if labels.ndim > 1 else labels.astype(int)
    top = np.argpartition(-np.asarray(pred), min(k, pred.shape[1]) - 1, axis=1)[:, :k]
    return float(np.mean((top == lab[:, None]).any(axis=1)))
