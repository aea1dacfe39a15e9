"""hostnet -- a TensorFlow-free stand-in for the small slice of Keras the GPFQ host code touches.

The reference's activation collection (`_get_layer_data_generator`, quantized_network.py:408-502) and
patch extraction (`_segment_data2D` :123-183) are host-side TensorFlow/Keras code that BASELINE.json's
north_star leaves on the host.  TensorFlow is not installed in this image, so this module provides the
closed API surface listed in SURVEY.md App. D with NumPy float32 forward passes:

    Sequential / Model(inputs=, outputs=) / clone_model, layers with .get_weights() .set_weights()
    .use_bias .input .output .input_shape .inbound_nodes[0].inbound_layers .strides .padding
    .dilation_rate and class names Dense, Conv2D, DepthwiseConv2D, BatchNormalization, MaxPooling2D,
    Flatten, Dropout, Activation, ReLU, InputLayer; `Sequence`; `extract_patches`.

It is host plumbing (random-init architectures of the reference's configs, forward passes to collect
layer inputs), not the hot path: the hot path runs in libgpfq.so.
"""
from __future__ import annotations

import copy
from math import ceil

import numpy as np


# ---------------------------------------------------------------------------------------------
# symbolic handles so that Model(inputs=net.layers[0].input, outputs=[layer.output]) works
# ---------------------------------------------------------------------------------------------
class KTensor:
    def __init__(self, layer, kind):
        self.layer, self.kind = layer, kind


class Node:
    def __init__(self, inbound_layers):
        self.inbound_layers = inbound_layers  # a single layer object, as Keras does for one input


def _act(name):
    if name in (None, "linear"):
        return lambda x: x
    if name == "relu":
        return lambda x: np.maximum(x, 0)
    if name == "softmax":
        def sm(x):
            e = np.exp(x - x.max(axis=-1, keepdims=True))
            return (e / e.sum(axis=-1, keepdims=True)).astype(np.float32)
        return sm
    if name == "sigmoid":
        return lambda x: (1 / (1 + np.exp(-x))).astype(np.float32)
    if name == "tanh":
        return np.tanh
    raise ValueError(f"activation {name!r} not supported by hostnet")


class Layer:
    use_bias = False

    def __init__(self, name=None, input_shape=None):
        self.name = name or self.__class__.__name__.lower()
        self._given_input_shape = tuple(input_shape) if input_shape is not None else None
        self.weights = []
        self.inbound_nodes = []
        self.input_shape = None
        self.output_shape = None
        self.model = None
        self.index = None

    # Keras surface -------------------------------------------------------------------------
    def get_weights(self):
        return [w.copy() for w in self.weights]

    def set_weights(self, ws):
        if len(ws) != len(self.weights):
            raise ValueError(f"{self.name}: expected {len(self.weights)} weight arrays, got {len(ws)}")
        new = []
        for old, w in zip(self.weights, ws):
            w = np.asarray(w)
            if w.shape != old.shape:
                raise ValueError(f"{self.name}: weight shape {w.shape} != {old.shape}")
            new.append(w.astype(np.float32))  # Keras casts to the variable dtype
        self.weights = new

    @property
    def input(self):
        return KTensor(self, "in")

    @property
    def output(self):
        return KTensor(self, "out")

    # subclass hooks --------------------------------------------------------------------------
    def build(self, in_shape, rng):
        self.input_shape = (None, *in_shape)
        out = self.compute_output_shape(in_shape)
        self.output_shape = (None, *out)
        return out

    def compute_output_shape(self, in_shape):
        return in_shape

    def call(self, x):
        return x


class InputLayer(Layer):
    pass


def _glorot(rng, shape, fan_in, fan_out):
    lim = np.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-lim, lim, shape).astype(np.float32)


def _he(rng, shape, fan_in):
    lim = np.sqrt(6.0 / fan_in)
    return rng.uniform(-lim, lim, shape).astype(np.float32)


class Dense(Layer):
    def __init__(self, units, activation=None, use_bias=True, kernel_initializer="glorot_uniform", **kw):
        super().__init__(kw.get("name"), kw.get("input_shape"))
        self.units, self.use_bias, self.activation = int(units), bool(use_bias), activation
        self.kernel_initializer = kernel_initializer

    def build(self, in_shape, rng):
        n_in = int(in_shape[-1])
        if self.kernel_initializer == "ones":
            k = np.ones((n_in, self.units), np.float32)
        elif self.kernel_initializer == "he_uniform":
            k = _he(rng, (n_in, self.units), n_in)
        else:
            k = _glorot(rng, (n_in, self.units), n_in, self.units)
        self.weights = [k] + ([rng.uniform(-0.05, 0.05, self.units).astype(np.float32)] if self.use_bias else [])
        return super().build(in_shape, rng)

    def compute_output_shape(self, in_shape):
        return (*in_shape[:-1], self.units)

    def call(self, x):
        y = x @ self.weights[0]
        if self.use_bias:
            y = y + self.weights[1]
        return _act(self.activation)(y).astype(np.float32)


def _same_pad(size, k_eff, stride):
    out = -(-size // stride)
    total = max((out - 1) * stride + k_eff - size, 0)
    return out, total // 2, total - total // 2


def extract_patches(images, sizes, strides, rates, padding):
    """NumPy equivalent of tf.image.extract_patches: (n, H, W, C) -> (n, Ho, Wo, kh*kw*C), depth order
    (row, col, channel).  Used at quantized_network.py:158-172 with C == 1."""
    images = np.asarray(images)
    n, H, W, C = images.shape
    kh, kw = int(sizes[1]), int(sizes[2])
    sh, sw = int(strides[1]), int(strides[2])
    rh, rw = int(rates[1]), int(rates[2])
    keh, kew = (kh - 1) * rh + 1, (kw - 1) * rw + 1
    if str(padding).upper() == "SAME":
        Ho, pt, pb = _same_pad(H, keh, sh)
        Wo, pl, pr = _same_pad(W, kew, sw)
        images = np.pad(images, ((0, 0), (pt, pb), (pl, pr), (0, 0)))
    else:
        Ho, Wo = (H - keh) // sh + 1, (W - kew) // sw + 1
    out = np.empty((n, Ho, Wo, kh * kw * C), dtype=images.dtype)
    for r in range(kh):
        for c in range(kw):
            blk = images[:, r * rh: r * rh + (Ho - 1) * sh + 1: sh, c * rw: c * rw + (Wo - 1) * sw + 1: sw, :]
            out[..., (r * kw + c) * C:(r * kw + c + 1) * C] = blk
    return out


class Conv2D(Layer):
    def __init__(self, filters, kernel_size, strides=(1, 1), padding="valid", dilation_rate=(1, 1), activation=None,
                 use_bias=True, kernel_initializer="he_uniform", groups=1, **kw):
        super().__init__(kw.get("name"), kw.get("input_shape"))
        # Keras' `groups`: input channels and filters split into `groups` groups, filters of group g see only the input channels
        # of group g; the kernel is (kh, kw, c_in // groups, filters)
        self.groups = int(groups)
        ks = (kernel_size, kernel_size) if np.isscalar(kernel_size) else tuple(kernel_size)
        self.filters, self.kernel_size = int(filters), (int(ks[0]), int(ks[1]))
        self.strides = (strides, strides) if np.isscalar(strides) else tuple(strides)
        self.dilation_rate = (dilation_rate, dilation_rate) if np.isscalar(dilation_rate) else tuple(dilation_rate)
        self.padding, self.activation, self.use_bias = padding, activation, bool(use_bias)
        self.kernel_initializer = kernel_initializer

    def _kernel_shape(self, c_in):
        if c_in % self.groups or self.filters % self.groups:
            raise ValueError(f"groups={self.groups} must divide the {c_in} input channels and the {self.filters} filters")
        return (*self.kernel_size, c_in // self.groups, self.filters)

    def build(self, in_shape, rng):
        c_in = int(in_shape[-1])
        shape = self._kernel_shape(c_in)
        fan_in = self.kernel_size[0] * self.kernel_size[1] * shape[2]
        k = _he(rng, shape, fan_in) if self.kernel_initializer == "he_uniform" else \
            _glorot(rng, shape, fan_in, self.kernel_size[0] * self.kernel_size[1] * self.filters)
        n_out = self._n_out(c_in)
        self.weights = [k] + ([rng.uniform(-0.05, 0.05, n_out).astype(np.float32)] if self.use_bias else [])
        return super().build(in_shape, rng)

    def _n_out(self, c_in):
        return self.filters

    def compute_output_shape(self, in_shape):
        H, W, C = in_shape
        keh = (self.kernel_size[0] - 1) * self.dilation_rate[0] + 1
        kew = (self.kernel_size[1] - 1) * self.dilation_rate[1] + 1
        if self.padding.lower() == "same":
            Ho, Wo = -(-H // self.strides[0]), -(-W // self.strides[1])
        else:
            Ho, Wo = (H - keh) // self.strides[0] + 1, (W - kew) // self.strides[1] + 1
        return (Ho, Wo, self._n_out(C))

    def _patches(self, x):
        return extract_patches(x, [1, *self.kernel_size, 1], [1, *self.strides, 1], [1, *self.dilation_rate, 1],
                               self.padding.upper())

    def call(self, x):
        p = self._patches(x)                                   # (n, Ho, Wo, kh*kw*C)
        if self.groups == 1:
            k = self.weights[0].reshape(-1, self.weights[0].shape[-1])  # (kh*kw*C, F)
            y = p.reshape(-1, p.shape[-1]) @ k
        else:
            kk, G = self.kernel_size[0] * self.kernel_size[1], self.groups
            Cg, F = self.weights[0].shape[2:]
            k = self.weights[0].reshape(kk, Cg, G, F // G)     # filter g*Fg + f of group g
            y = np.einsum("ptgc,tcgf->pgf", p.reshape(-1, kk, G, Cg), k).reshape(-1, F)
        y = y.reshape(*p.shape[:3], -1)
        if self.use_bias:
            y = y + self.weights[1]
        return _act(self.activation)(y).astype(np.float32)


class DepthwiseConv2D(Conv2D):
    def __init__(self, kernel_size, strides=(1, 1), padding="valid", depth_multiplier=1, dilation_rate=(1, 1),
                 activation=None, use_bias=True, **kw):
        super().__init__(depth_multiplier, kernel_size, strides, padding, dilation_rate, activation, use_bias, **kw)
        self.depth_multiplier = int(depth_multiplier)

    def _kernel_shape(self, c_in):
        return (*self.kernel_size, c_in, self.depth_multiplier)

    def _n_out(self, c_in):
        return c_in * self.depth_multiplier

    def call(self, x):
        n, H, W, C = x.shape
        kh, kw = self.kernel_size
        p = self._patches(x)
        Ho, Wo = p.shape[1], p.shape[2]
        p = p.reshape(n, Ho, Wo, kh * kw, C)
        k = self.weights[0].reshape(kh * kw, C, self.depth_multiplier)
        y = np.einsum("nhwtc,tcd->nhwcd", p, k).reshape(n, Ho, Wo, C * self.depth_multiplier)
        if self.use_bias:
            y = y + self.weights[1]
        return _act(self.activation)(y).astype(np.float32)


class BatchNormalization(Layer):
    def __init__(self, epsilon=1e-3, **kw):
        super().__init__(kw.get("name"))
        self.epsilon = epsilon

    def build(self, in_shape, rng):
        c = int(in_shape[-1])
        # a "trained" normaliser: non-trivial statistics so the quantized twin's inputs differ meaningfully
        self.weights = [rng.uniform(0.8, 1.2, c).astype(np.float32), rng.uniform(-0.1, 0.1, c).astype(np.float32),
                        rng.uniform(-0.1, 0.1, c).astype(np.float32), rng.uniform(0.5, 1.5, c).astype(np.float32)]
        return super().build(in_shape, rng)

    def call(self, x):
        g, b, mu, var = self.weights
        return ((x - mu) / np.sqrt(var + np.float32(self.epsilon)) * g + b).astype(np.float32)


class MaxPooling2D(Layer):
    def __init__(self, pool_size=(2, 2), strides=None, padding="valid", **kw):
        super().__init__(kw.get("name"))
        self.pool_size = (pool_size, pool_size) if np.isscalar(pool_size) else tuple(pool_size)
        self.strides = self.pool_size if strides is None else ((strides, strides) if np.isscalar(strides) else tuple(strides))
        self.padding = padding

    def compute_output_shape(self, in_shape):
        H, W, C = in_shape
        return ((H - self.pool_size[0]) // self.strides[0] + 1, (W - self.pool_size[1]) // self.strides[1] + 1, C)

    def call(self, x):
        n, H, W, C = x.shape
        ph, pw = self.pool_size
        sh, sw = self.strides
        Ho, Wo = (H - ph) // sh + 1, (W - pw) // sw + 1
        out = np.full((n, Ho, Wo, C), -np.inf, dtype=np.float32)
        for r in range(ph):
            for c in range(pw):
                out = np.maximum(out, x[:, r: r + (Ho - 1) * sh + 1: sh, c: c + (Wo - 1) * sw + 1: sw, :])
        return out


class Flatten(Layer):
    def compute_output_shape(self, in_shape):
        return (int(np.prod(in_shape)),)

    def call(self, x):
        return x.reshape(x.shape[0], -1)


class Dropout(Layer):
    def __init__(self, rate=0.5, **kw):
        super().__init__(kw.get("name"))
        self.rate = rate


class Activation(Layer):
    def __init__(self, activation, **kw):
        super().__init__(kw.get("name"))
        self.activation = activation

    def call(self, x):
        return _act(self.activation)(x).astype(np.float32)


class ReLU(Activation):
    def __init__(self, **kw):
        super().__init__("relu", **kw)


# ---------------------------------------------------------------------------------------------
# models
# ---------------------------------------------------------------------------------------------
class Sequential:
    def __init__(self, layers=None, input_shape=None, seed=0, name="sequential"):
        self.name = name
        self.layers = []
        self._seed = seed
        self._input_shape = tuple(input_shape) if input_shape is not None else None
        self.built = False
        for l in (layers or []):
            self.add(l)
        if self._input_shape is not None and self.layers:
            self.build(self._input_shape)

    def add(self, layer):
        if not self.layers and layer._given_input_shape is not None and self._input_shape is None:
            self._input_shape = layer._given_input_shape
        self.layers.append(layer)
        self.built = False

    def build(self, input_shape=None, seed=None):
        if input_shape is not None:
            self._input_shape = tuple(input_shape)
        if self._input_shape is None:
            raise ValueError("input shape unknown")
        rng = np.random.default_rng(self._seed if seed is None else seed)
        shape = self._input_shape
        prev = None
        for i, l in enumerate(self.layers):
            l.model, l.index = self, i
            l.inbound_nodes = [Node(prev)] if prev is not None else []
            shape = l.build(shape, rng)
            prev = l
        self.built = True
        return self

    def _ensure(self):
        if not self.built:
            self.build()

    def get_weights(self):
        self._ensure()
        return [w for l in self.layers for w in l.get_weights()]

    def set_weights(self, ws):
        self._ensure()
        ws, k = list(ws), 0
        for l in self.layers:
            n = len(l.weights)
            l.set_weights(ws[k:k + n])
            k += n

    def run(self, x, first=0, last=None):
        """Outputs of layers first..last (inclusive) applied in order."""
        self._ensure()
        x = np.asarray(x, dtype=np.float32)
        for l in self.layers[first:(len(self.layers) if last is None else last + 1)]:
            x = l.call(x)
        return x

    def predict_on_batch(self, x):
        return self.run(x)

    def predict(self, x, batch_size=256, verbose=0):
        x = np.asarray(x)
        return np.concatenate([self.run(x[i:i + batch_size]) for i in range(0, len(x), batch_size)])

    def evaluate(self, x, y, batch_size=256, verbose=0):
        """(loss, accuracy) with sparse or one-hot labels, softmax outputs assumed."""
        p = self.predict(x, batch_size)
        y = np.asarray(y)
        lab = y.argmax(-1) if y.ndim > 1 and y.shape[-1] > 1 else y.reshape(-1).astype(int)
        acc = float(np.mean(p.argmax(-1) == lab))
        loss = float(-np.mean(np.log(np.maximum(p[np.arange(len(lab)), lab], 1e-30))))
        return loss, acc


class Model:
    """Model(inputs=net.layers[0].input, outputs=[layer.output, ...]) -- partial forward models (:459-462)."""

    def __init__(self, inputs, outputs):
        outs = outputs if isinstance(outputs, (list, tuple)) else [outputs]
        self._single = len(outs) == 1
        self._net = inputs.layer.model
        self._first = inputs.layer.index
        self._lasts = [o.layer.index if o.kind == "out" else o.layer.index - 1 for o in outs]

    def predict_on_batch(self, x):
        res = [self._net.run(x, self._first, last) for last in self._lasts]
        return res[0] if self._single else res


def clone_model(net):
    """Same architecture, freshly initialised weights (the reference copies the weights right after, :377-380)."""
    new = Sequential(name=net.name + "_clone", seed=net._seed + 1)
    for l in net.layers:
        c = copy.copy(l)
        c.weights = []
        c.inbound_nodes = []
        new.add(c)
    new.build(net._input_shape)
    return new


class Sequence:
    """keras.utils.Sequence base class."""

    def __len__(self):
        raise NotImplementedError

    def __getitem__(self, idx):
        raise NotImplementedError


class ArraySequence(Sequence):
    """The reference's MNISTSequence / CIFAR10Sequence (quantized_network.py:235-293): slice batches of an array."""

    def __init__(self, x_set, y_set, batch_size):
        self.x, self.y, self.batch_size = x_set, y_set, batch_size

    def __len__(self):
        return ceil(len(self.x) / self.batch_size)

    def __getitem__(self, idx):
        sl = slice(idx * self.batch_size, (idx + 1) * self.batch_size)
        return np.array(self.x[sl]), np.array(self.y[sl])


# ---------------------------------------------------------------------------------------------
# the reference's architectures, random-init (there are no datasets or checkpoints offline)
# ---------------------------------------------------------------------------------------------
def mnist_mlp(seed=0, widths=(500, 300), n_in=784, n_out=10):
    """train_mnist_mlp.py:61-73 -- Flatten, Dense+BN (relu) x2, Dense softmax."""
    layers = [Flatten()]
    for w in widths:
        layers += [Dense(w, activation="relu", kernel_initializer="glorot_uniform"), BatchNormalization()]
    layers += [Dense(n_out, activation="softmax")]
    side = int(round(np.sqrt(n_in)))
    return Sequential(layers, input_shape=(side, side) if side * side == n_in else (n_in,), seed=seed)


def cifar10_cnn(seed=0, size=32, widths=(32, 64, 128), dense=128, n_out=10):
    """train_cifar10_cnn.py:63-88 -- three [Conv-BN-Conv-BN-Pool-Dropout] blocks, Flatten, Dense-BN-Dropout, Dense."""
    layers = []
    for w in widths:
        layers += [Conv2D(w, 3, padding="same", activation="relu"), BatchNormalization(),
                   Conv2D(w, 3, padding="same", activation="relu"), BatchNormalization(),
                   MaxPooling2D(2), Dropout(0.2)]
    layers += [Flatten(), Dense(dense, activation="relu", kernel_initializer="he_uniform"), BatchNormalization(),
               Dropout(0.5), Dense(n_out, activation="softmax")]
    return Sequential(layers, input_shape=(size, size, 3), seed=seed)


def vgg16_like(seed=0, size=224, scale=1, n_out=1000, fc=4096):
    """Keras VGG16 (quantize_pretrained_imagenet.py:43,89): InputLayer, 13 conv 3x3 'same' relu, 5 pools, fc1 fc2 predictions.
    `scale` divides the channel counts (tests use a thin copy)."""
    cfg = [(64, 2), (128, 2), (256, 3), (512, 3), (512, 3)]
    layers = [InputLayer()]
    for c, reps in cfg:
        layers += [Conv2D(max(c // scale, 1), 3, padding="same", activation="relu") for _ in range(reps)]
        layers += [MaxPooling2D(2)]
    layers += [Flatten(), Dense(fc, activation="relu"), Dense(fc, activation="relu"), Dense(n_out, activation="softmax")]
    return Sequential(layers, input_shape=(size, size, 3), seed=seed)
