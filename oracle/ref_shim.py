"""TEST INFRASTRUCTURE ONLY -- loader for the *unmodified* reference module.

The reference (`$GPFQ_REFERENCE_ROOT/scripts/quantized_network.py`) imports TensorFlow and
h5py at module scope (`:21-25`, `:31`); neither is installed here.  The arithmetic of
the hot path (`_bit_round_parallel :40`, `_quantize_weight_parallel :59`,
`_quantize_neuron_parallel :91`, `_quantize_filter2D_parallel_jit :185`) only needs
NumPy + SciPy.  This shim registers empty stand-in modules for the TensorFlow names
and an in-memory `h5py.File` (a dict of ndarrays behind a context manager), then
imports the reference file from where it lies.  Nothing of the reference is copied.

The reference is not part of this repository: set GPFQ_REFERENCE_ROOT to a checkout of
elybrand/quantized_neural_networks to use it.  This module is used by
`oracle/make_golden.py` (fixture generation) and by the tests that run the reference
itself (they skip when GPFQ_REFERENCE_ROOT is unset).
"""
from __future__ import annotations

import importlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("GPFQ_REFERENCE_ROOT", "")
_SCRIPTS = os.path.join(REFERENCE_ROOT, "scripts")

# name -> {dataset -> ndarray}; the reference passes file *names* to its workers.
MEMORY_FILES: dict[str, dict] = {}


class _MemDataset:
    """Stand-in for an h5py dataset: float32, zero-filled, basic / ellipsis slicing, `resize(n, axis)` (the calls the
    reference makes: quantized_network.py:118-119, :487-495, :769-770, :789-797)."""

    def __init__(self, arr):
        self._a = arr

    @property
    def shape(self):
        return self._a.shape

    def __getitem__(self, key):
        return self._a[key]

    def __setitem__(self, key, value):
        self._a[key] = value

    def __array__(self, dtype=None, copy=None):
        return self._a if dtype is None else self._a.astype(dtype)

    def resize(self, size, axis=None):
        import numpy as np
        shape = list(self._a.shape)
        if axis is None:
            shape = list(size)
        else:
            shape[axis] = int(size)
        new = np.zeros(shape, dtype=self._a.dtype)
        keep = tuple(slice(0, min(a, b)) for a, b in zip(self._a.shape, shape))
        new[keep] = self._a[keep]
        self._a = new


class _MemGroup(dict):
    """What `with h5py.File(...) as hf` yields: a mapping of datasets plus `create_dataset`."""

    def create_dataset(self, name, shape=None, data=None, dtype=None, **kw):
        import numpy as np
        if data is not None:
            arr = np.array(data, dtype=np.float32 if dtype is None else dtype)   # h5py keeps the dtype of `data`
            if dtype is None and hasattr(data, "dtype"):
                arr = np.array(data, dtype=data.dtype)
        else:
            arr = np.zeros(shape, dtype=np.float32 if dtype is None else dtype)  # h5py default dtype is float32 ('f')
        self[name] = _MemDataset(arr)
        return self[name]


class _MemFile:
    """Stand-in for h5py.File: 'w' creates/clears a named group, 'r' opens it.  A zero-byte file of the same name is left
    in the working directory because the reference removes its hand-off files with os.remove (:574, :725, :867)."""

    def __init__(self, name, mode="r"):
        key = os.path.basename(str(name))
        if mode == "w":
            MEMORY_FILES[key] = _MemGroup()
            try:
                open(str(name), "a").close()
            except OSError:
                pass
        self._d = MEMORY_FILES[key]

    def __enter__(self):
        return self._d

    def __exit__(self, *exc):
        return False


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(_SCRIPTS, "quantized_network.py"))


def load():
    """Import and return the reference `quantized_network` module (unmodified)."""
    if "quantized_network" in sys.modules and getattr(
        sys.modules["quantized_network"], "__gpfq_shim__", False
    ):
        return sys.modules["quantized_network"]
    if not available():
        raise FileNotFoundError(f"reference not present under GPFQ_REFERENCE_ROOT={REFERENCE_ROOT!r}")

    def mod(name, **attrs):
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    def _absent(*a, **k):
        raise RuntimeError("TensorFlow is not installed; this TensorFlow call has no stand-in")

    # The Keras / TensorFlow names the reference's HOST code touches (SURVEY.md App. D) map to the NumPy stand-ins of
    # quantized_neural_networks_b200.hostnet, so that `QuantizedNeuralNetwork(...).quantize_network()` (:576-590),
    # `_get_layer_data_generator` (:408-502) and `_build_patch_array` (:729-809) run UNMODIFIED from the reference file.
    from quantized_neural_networks_b200 import hostnet
    Sequence = hostnet.Sequence

    def extract_patches(images, sizes, strides, rates, padding):
        return hostnet.extract_patches(images, sizes, strides, rates, padding)

    saved = {k: sys.modules.get(k) for k in (
        "tensorflow", "tensorflow.keras", "tensorflow.keras.utils", "tensorflow.keras.backend",
        "tensorflow.keras.models", "tensorflow.image", "h5py")}
    tf = mod("tensorflow", convert_to_tensor=_absent)
    keras = mod("tensorflow.keras")
    tf.keras = keras
    keras.utils = mod("tensorflow.keras.utils", Sequence=Sequence)
    keras.backend = mod("tensorflow.keras.backend", function=_absent)
    keras.models = mod("tensorflow.keras.models", Model=hostnet.Model, clone_model=hostnet.clone_model)
    tf.image = mod("tensorflow.image", extract_patches=extract_patches)
    mod("h5py", File=_MemFile)

    sys.path.insert(0, _SCRIPTS)
    try:
        ref = importlib.import_module("quantized_network")
    finally:
        sys.path.remove(_SCRIPTS)
        # leave the stubs only inside the imported module's namespace
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    ref.__gpfq_shim__ = True
    return ref


def ref_quantize_neuron(w, X, Xq, alphabet):
    """Run the reference's `_quantize_neuron_parallel` (:91-121) on in-memory data.

    X, Xq: float32 (N0, m) feature-major, exactly the `wX`/`qX` datasets of `:469-492`.
    """
    ref = load()
    name = f"layer_mem_{os.getpid()}_{id(X)}.h5"
    MEMORY_FILES[name] = {"wX": X, "qX": Xq}
    try:
        return ref._quantize_neuron_parallel(w, name, alphabet)
    finally:
        MEMORY_FILES.pop(name, None)


def ref_quantize_filter(chan_filter, Xp, Xqp, alphabet, channel_idx=0):
    """Run the reference's `_quantize_filter2D_parallel_jit` (:185-233) on in-memory patches."""
    ref = load()
    name = f"channel_mem_{os.getpid()}_{id(Xp)}.h5"
    MEMORY_FILES[name] = {f"wX_channel{channel_idx}": Xp, f"qX_channel{channel_idx}": Xqp}
    try:
        return ref._quantize_filter2D_parallel_jit(chan_filter, channel_idx, name, alphabet)
    finally:
        MEMORY_FILES.pop(name, None)


class SerialExecutor:
    """Drop-in for concurrent.futures.ProcessPoolExecutor that runs every task at submit time in this process: the
    reference's fan-out (:549-567, :706-721) only needs submit / as_completed / the context manager.  (A forked pool works
    too -- the in-memory files are inherited -- but a serial run is deterministic and cannot hang on threaded BLAS.)"""

    def __init__(self, *a, **k):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False

    def submit(self, fn, *args, **kwargs):
        import concurrent.futures
        fut = concurrent.futures.Future()
        try:
            fut.set_result(fn(*args, **kwargs))
        except BaseException as exc:   # noqa: BLE001 -- handed to the caller through the future, as a pool would
            fut.set_exception(exc)
        return fut


class serial_pool:
    """Context manager: concurrent.futures.ProcessPoolExecutor -> SerialExecutor while the reference's methods run."""

    def __enter__(self):
        import concurrent.futures
        self._saved = concurrent.futures.ProcessPoolExecutor
        concurrent.futures.ProcessPoolExecutor = SerialExecutor
        return self

    def __exit__(self, *exc):
        import concurrent.futures
        concurrent.futures.ProcessPoolExecutor = self._saved
        return False
