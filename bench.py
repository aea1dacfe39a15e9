#!/usr/bin/env python
"""bench.py -- GPFQ hot path on B200: quantized weights/s of a full-network pass (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py ... --dump-outputs DIR                   # + every layer's Q of the last timed step, DIR/<layer>.npy
    python bench.py --impl reference --gpus N --steps K ...  # the reference's NumPy path on the host cores

Default workload (config.workload): BASELINE.json configs[2], the north-star target -- a VGG16-shaped full-network GPFQ
ternary pass (quantize_pretrained_imagenet.py:43-50: ternary, 1504 images): thirteen 3x3 'same' Conv2D layers handed over
as their NHWC activation tensors (what _get_layer_data_generator collects, quantized_network.py:468; 109 GB resident) and
three Dense layers (25088->4096->4096->1000, m = 1504), synthetic activations (SURVEY.md 8d), random-init weights.
One "step" = one pass of the hot path over all sixteen layers.  --workload cifar10_cnn | mnist_mlp | dense_sweep run
BASELINE configs[1], [0] and [3] the same way (configs[4], the 20-alphabet grid: tools/grid_bench.py).

  value     whole-job weights/s with every input resident in HBM when the timed region starts (CUDA events on the
            launching stream, max over ranks).  N > 1: conv layers are split over IMAGES (each rank contracts its
            n_img / N images of every channel, one NCCL all-reduce of the per-channel 9 x 9 Grams, every rank walks every
            channel), Dense neurons are sharded with the inputs replicated and the Q blocks all-gathered (fp32, what
            Keras set_weights stores) -- all of it inside the timed region.  Total work is fixed => "strong".
  e2e       the same pass through the reference-facing C ABI with HOST (pinned) buffers, layer by layer: H2D copies,
            kernels and the D2H copy of Q inside the timed region (host wall clock around the synchronous calls).
  per_layer every layer's time, weights/s and fraction of its governing roofline (conv: fp64 DFMA pipe / HBM; Dense: the
            stage that takes the most time).
  roofline  the kernel that takes the largest share of the step.
  parity    (N = 1) the literal C oracle run on a sample of neurons / filters of EVERY layer at full size, on the very host
            buffers the e2e leg hands to the C ABI, compared with the Q the C ABI returned: agreement, relative-residual
            delta, entries checked.  The run fails below 99.99 % / above 1e-6.
  cpu_baseline  the oracle's NumPy restatement of the reference walk (kind "port": the reference is Python and does not
            travel to the GPU box), one process per host core like the reference's ProcessPoolExecutor, on a bounded
            sample of every layer (conv layers: one channel, `cores` filters, a subset of the images), extrapolated
            linearly in filters x channels x images / neurons.
"""
from __future__ import annotations

import os

os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")   # the CPU-baseline workers are one process per core (SURVEY.md 8d)
os.environ.setdefault("OMP_NUM_THREADS", "1")

import argparse
import json
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DFMA_RATE = 17.05e12     # DFMA / s, measured on this pool's B200 (profiles/fp64_pipes_r1.txt)
DMMA_RATE = 18.55e12     # fp64 MACs / s through DMMA.8x8x4 (same pipe)
DUMP_BYTES = 60_000_000  # --dump-outputs payload over all layers: under 64 MB with the .npy headers


def conv(name, C, F, H):
    return dict(name=name, kind="conv", C=C, F=F, H=H)


def dense(name, N0, N1, m=None):
    return dict(name=name, kind="dense", N0=N0, N1=N1, m=m)


# SURVEY.md App. B.  VGG16: Keras VGG16() as instantiated by quantize_pretrained_imagenet.py:43,89
VGG_LAYERS = [conv("conv0", 3, 64, 224), conv("conv1", 64, 64, 224), conv("conv2", 64, 128, 112), conv("conv3", 128, 128, 112),
              conv("conv4", 128, 256, 56), conv("conv5", 256, 256, 56), conv("conv6", 256, 256, 56), conv("conv7", 256, 512, 28),
              conv("conv8", 512, 512, 28), conv("conv9", 512, 512, 28), conv("conv10", 512, 512, 14), conv("conv11", 512, 512, 14),
              conv("conv12", 512, 512, 14), dense("fc1", 25088, 4096), dense("fc2", 4096, 4096), dense("fc3", 4096, 1000)]
CIFAR_LAYERS = [conv("conv0", 3, 32, 32), conv("conv2", 32, 32, 32), conv("conv6", 32, 64, 16), conv("conv8", 64, 64, 16),
                conv("conv12", 64, 128, 8), conv("conv14", 128, 128, 8), dense("dense19", 2048, 128), dense("dense22", 128, 10)]
MNIST_LAYERS = [dense("dense1", 784, 500), dense("dense3", 500, 300), dense("dense5", 300, 10)]
SWEEP_LAYERS = [dense(f"dense_{n}_{m // 1000}k", n, n, m) for n in (1024, 4096, 16384) for m in (5000, 25000, 100000)]

WORKLOADS = {
    "vgg16": dict(layers=VGG_LAYERS, n_img=1504, bits=np.log2(3), c=3,
                  desc="VGG16 (BASELINE configs[2]): 13x Conv2D 3x3 'same' from NHWC activations + Dense 25088->4096->4096->1000, "
                       "ternary (quantize_pretrained_imagenet.py:43-50)",
                  l2="109 GB of layer inputs per pass stream through HBM between two uses of any buffer; no flush needed"),
    "cifar10_cnn": dict(layers=CIFAR_LAYERS, n_img=5008, bits=4, c=4,
                        desc="CIFAR10 CNN (BASELINE configs[1]): 6x Conv2D 3x3 from NHWC activations + Dense 2048->128->10, 4-bit",
                        l2="2.9 GB of layer inputs per pass exceed the 126 MB L2; no flush needed"),
    "mnist_mlp": dict(layers=MNIST_LAYERS, n_img=25000, bits=np.log2(3), c=3,
                      desc="MNIST MLP 784-500-300-10 (BASELINE configs[0]), ternary, m = 25000",
                      l2="240 MB of layer inputs per pass exceed the 126 MB L2; no flush needed"),
    "dense_sweep": dict(layers=SWEEP_LAYERS, n_img=0, bits=np.log2(3), c=3,
                        desc="synthetic Dense sweep (BASELINE configs[3]): N0 = N1 in {1024, 4096, 16384} x m in {5k, 25k, 100k}, ternary",
                        l2="28 GB of layer inputs per pass exceed L2; no flush needed"),
}


def shard_range(n, rank, world):
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def layer_weights(l):
    return 9 * l["C"] * l["F"] if l["kind"] == "conv" else l["N0"] * l["N1"]


def make_alphabet(W_abs_median, wl):
    """rad * linspace(-1, 1, K) (quantized_network.py:396, :544-545)."""
    return wl["c"] * float(W_abs_median) * np.linspace(-1, 1, int(round(2 ** wl["bits"])))


# ----------------------------------------------------------------------------------------------------------------
# synthetic data (device side; torch is only the buffer / generator)
# ----------------------------------------------------------------------------------------------------------------
def build_device_inputs(wl, n_img, rank, world, dev):
    """Per layer a dict of device tensors.  conv: NHWC activations act / actq of THIS RANK's images (the image split of a
    multi-GPU job; all images when world == 1); dense: (N0, m) X / Xq replicated, neurons j0..j1 are this rank's."""
    import torch
    out = []
    for li, l in enumerate(wl["layers"]):
        g = torch.Generator(device=dev).manual_seed(1000 + li)
        first = li == 0 and wl is not WORKLOADS["dense_sweep"]
        if l["kind"] == "conv":
            C, F, H = l["C"], l["F"], l["H"]
            W = (torch.rand((3, 3, C, F), device=dev, generator=g) * 2 - 1) * float(np.sqrt(6.0 / (9 * C)))
            A = make_alphabet(torch.median(W.abs().flatten()), wl)
            lo, hi = shard_range(n_img, rank, world)
            g.manual_seed(1000 + li + 7919 * (rank + 1))
            shape = (hi - lo, H, H, C)
            act = torch.empty(shape, device=dev)
            actq = None if first else torch.empty(shape, device=dev)
            step = max(1, int(2 ** 28 // (H * H * C)))      # chunked: temporaries of a 19 GB randn would double the footprint
            for i0 in range(0, hi - lo, step):
                n = min(step, hi - lo - i0)
                if first:   # image-like input, X == Xq
                    z = torch.rand((n, H, H, C), device=dev, generator=g)
                    if wl is not WORKLOADS["vgg16"]:    # MNIST / CIFAR-like sparsity (SURVEY.md 8d)
                        z = z * (torch.rand((n, H, H, C), device=dev, generator=g) < 0.5)
                    act[i0:i0 + n] = z
                else:       # hidden: X = relu(Z), Xq = relu(Z + 0.05 N)
                    z = torch.randn((n, H, H, C), device=dev, generator=g)
                    act[i0:i0 + n] = torch.relu(z)
                    actq[i0:i0 + n] = torch.relu(z + 0.05 * torch.randn((n, H, H, C), device=dev, generator=g))
                del z
            out.append(dict(l, W=W, A=A, act=act, actq=actq, first=first, img_lo=lo, img_hi=hi, n_img=n_img,
                            out=torch.zeros((1, 3, 3, C, F), dtype=torch.float64, device=dev)))
        else:
            N0, N1 = l["N0"], l["N1"]
            m = l["m"] or n_img
            W = (torch.rand((N0, N1), device=dev, generator=g) * 2 - 1) * float(np.sqrt(6.0 / N0))
            A = make_alphabet(torch.median(W.abs().flatten()), wl)
            X = torch.empty((N0, m), device=dev)
            Xq = None if first else torch.empty((N0, m), device=dev)
            step = max(1, int(2 ** 28 // m))
            for t0 in range(0, N0, step):
                n = min(step, N0 - t0)
                if first:
                    X[t0:t0 + n] = torch.rand((n, m), device=dev, generator=g) * (torch.rand((n, m), device=dev, generator=g) < 0.5)
                else:
                    z = torch.randn((n, m), device=dev, generator=g)
                    X[t0:t0 + n] = torch.relu(z)
                    Xq[t0:t0 + n] = torch.relu(z + 0.05 * torch.randn((n, m), device=dev, generator=g))
                    del z
            lo, hi = shard_range(N1, rank, world)
            d = dict(l, W=W, A=A, X=X, Xq=Xq, j0=lo, j1=hi, m=m, first=first,
                     out=torch.zeros((1, N0, N1), dtype=torch.float64, device=dev))
            if world > 1:   # Q exchange buffers (fp32, what set_weights stores): equal-width column blocks
                width = -(-N1 // world)
                d["gblk"] = torch.zeros((N0, width), dtype=torch.float32, device=dev)
                d["gout"] = torch.empty((world, N0, width), dtype=torch.float32, device=dev)
            out.append(d)
        torch.cuda.empty_cache()
    return out


def api_calls(d, world):
    return 2 if (d["kind"] == "conv" and world > 1) else 1


def run_layer_device(eng, d, world):
    """One layer of the device-resident pass (asynchronous on torch's current stream)."""
    import torch.distributed as dist
    if d["kind"] == "conv":
        if world > 1:
            gram = eng.conv_gram_nhwc(d["act"], d["actq"], (3, 3), sync=False)
            dist.all_reduce(gram)
            eng.conv_layer_from_gram(gram, d["W"], d["A"], out=d["out"], sync=False)
        else:
            eng.conv_layer_nhwc(d["act"], d["actq"], d["W"], d["A"], out=d["out"], sync=False)
    else:
        eng.dense_layer(d["X"], d["Xq"], d["W"], d["A"], j0=d["j0"], j1=d["j1"], out=d["out"], sync=False)
        if world > 1:
            d["gblk"][:, :d["j1"] - d["j0"]].copy_(d["out"][0][:, d["j0"]:d["j1"]])
            dist.all_gather_into_tensor(d["gout"], d["gblk"])


def layer_output(d, world):
    """The quantized kernel Q a caller holds after one layer of the device-resident pass: (3, 3, C, F) or (N0, N1)."""
    import torch
    if d["kind"] == "dense" and world > 1:     # the all-gathered column blocks, each trimmed to its rank's width
        blocks = [shard_range(d["N1"], r, world) for r in range(world)]
        return torch.cat([d["gout"][r][:, :hi - lo] for r, (lo, hi) in enumerate(blocks)], dim=1)
    return d["out"][0]


def dump_outputs(out_dir, data, world):
    """Writes every layer's Q of the last pass as out_dir/<layer>.npy (float64).  A layer with more entries than its share
    of DUMP_BYTES is written as a fixed sample: the entries at sorted random flat indices drawn from a generator seeded with
    the layer's index, so two runs with the same arguments write the same positions."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // 8 // len(data)
    for li, d in enumerate(data):
        Q = layer_output(d, world)
        if Q.numel() > cap:
            idx = np.sort(np.random.default_rng(li).choice(Q.numel(), cap, replace=False))
            Q = Q.reshape(-1)[torch.from_numpy(idx).to(Q.device)]
        np.save(os.path.join(out_dir, d["name"] + ".npy"), Q.to(torch.float64).cpu().numpy())


# ----------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            time.sleep(0.3)   # nvidia-smi needs a moment before its first sample
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# CPU side: the oracle.  A pool of one worker process per core, forked BEFORE CUDA is initialised; the sample of a layer
# reaches the workers as .npy files they memory-map (the reference hands its workers an HDF5 file name the same way).
# ----------------------------------------------------------------------------------------------------------------
_MM = {}


def _cpu_unit(args):
    tag, j = args
    from oracle import gpfq_oracle as O
    if _MM.get("tag") != tag:
        _MM.clear()
        _MM.update(tag=tag, W=np.load(tag + "_W.npy", mmap_mode="r"), X=np.load(tag + "_X.npy", mmap_mode="r"),
                   A=np.load(tag + "_A.npy"))
        _MM["Xq"] = np.load(tag + "_Xq.npy", mmap_mode="r") if os.path.exists(tag + "_Xq.npy") else _MM["X"]
    return O.quantize_neuron(np.asarray(_MM["W"][:, j]), _MM["X"], _MM["Xq"], _MM["A"])


def _cpu_noop(_):
    return os.getpid()


class CpuPool:
    def __init__(self, cores):
        import concurrent.futures as cf
        import multiprocessing as mp
        self.cores = cores
        base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > (2 << 30) else None
        self.dir = tempfile.mkdtemp(prefix="gpfq_bench_", dir=base)
        self.ex = cf.ProcessPoolExecutor(max_workers=cores, mp_context=mp.get_context("fork"))
        list(self.ex.map(_cpu_noop, range(4 * cores)))   # start every worker now
        self.n = 0

    def time_units(self, W, X, Xq, A, units):
        """Walks neurons `units` of the (N0, N1) problem (W, X, Xq) on the pool; returns (seconds, Q columns)."""
        self.n += 1
        tag = os.path.join(self.dir, f"s{self.n}")
        np.save(tag + "_W.npy", np.ascontiguousarray(W, dtype=np.float32))
        np.save(tag + "_X.npy", np.ascontiguousarray(X, dtype=np.float32))
        if Xq is not None and Xq is not X:
            np.save(tag + "_Xq.npy", np.ascontiguousarray(Xq, dtype=np.float32))
        np.save(tag + "_A.npy", np.asarray(A, dtype=np.float64))
        t0 = time.perf_counter()
        cols = list(self.ex.map(_cpu_unit, [(tag, int(j)) for j in units]))
        dt = time.perf_counter() - t0
        for f in os.listdir(self.dir):
            if f.startswith(f"s{self.n}_"):
                os.remove(os.path.join(self.dir, f))
        return dt, cols

    def close(self):
        self.ex.shutdown(wait=True, cancel_futures=True)
        shutil.rmtree(self.dir, ignore_errors=True)


def plane_patches(plane):
    """(9, n) patch matrix of one channel plane (n_img, H, H): 3x3 'same' stride 1, row r*3+c, patches in image-major
    order -- what _build_patch_array writes to channel{c}_patch_array.h5 (quantized_network.py:789-797)."""
    n_img, H = plane.shape[0], plane.shape[1]
    p = np.zeros((n_img, H + 2, H + 2), np.float32)
    p[:, 1:-1, 1:-1] = plane
    cols = np.empty((9, n_img * H * H), np.float32)
    for r in range(3):
        for cc in range(3):
            cols[r * 3 + cc] = p[:, r:r + H, cc:cc + H].reshape(-1)
    return cols


def cpu_time_layer(pool, l, W, A, planes=None, X=None, Xq=None, max_patches=600_000):
    """NumPy port of the reference walk on a bounded sample of layer `l`; returns (extrapolated seconds for the whole layer
    on pool.cores processes, weights actually walked, description).  conv: `planes` = (plane, planeq or None) of ONE
    channel, (n_img, H, H); the first images up to ~max_patches patch columns, `cores` filters; cost is linear in patch
    columns, filters and channels.  dense: 2 x cores neurons at full size; linear in neurons."""
    cores = pool.cores
    if l["kind"] == "conv":
        plane, planeq = planes
        n_img, H = plane.shape[0], plane.shape[1]
        n_s = max(1, min(n_img, max_patches // (H * H)))
        Xp = plane_patches(plane[:n_s])
        Xqp = Xp if planeq is None else plane_patches(planeq[:n_s])
        take = min(l["F"], cores)
        Wc = np.ascontiguousarray(W.reshape(9, -1)[:, :take])
        dt, _ = pool.time_units(Wc, Xp, Xqp, A, range(take))
        scale = (l["n_img_total"] / n_s) * (l["C"] * l["F"] / take)
        return dt * scale, 9 * take, f"{l['name']}:{take}f/{l['C'] * l['F']}x{n_s}img/{l['n_img_total']}"
    N1 = W.shape[1]
    take = min(N1, 2 * cores if l["N0"] >= 1024 else 4 * cores)
    dt, _ = pool.time_units(W[:, :take], X, Xq, A, range(take))
    return dt * (l["N1"] / take), l["N0"] * take, f"{l['name']}:{take}n/{l['N1']}"


def residual_rel(W, Q, X, Xq):
    """||X^T w - Xq^T q|| / ||X^T w|| per column (fp64)."""
    Xd, Xqd = np.asarray(X, dtype=np.float64), np.asarray(Xq, dtype=np.float64)
    a = Xd.T @ np.asarray(W, dtype=np.float64)
    r = a - Xqd.T @ Q
    return np.linalg.norm(r, axis=0) / np.maximum(np.linalg.norm(a, axis=0), 1e-300)


def parity_layer(l, W, A, Qgpu, X, Xq, units, cores):
    """Literal C oracle (oracle/gpfq_oracle.c, quantized_network.py:91-121 / :185-233) on columns `units` of the (N0, N1)
    problem at FULL size vs the same columns of the GPU result.  Returns the parity record of the layer."""
    from oracle import c_oracle
    units = list(units)
    Ws = np.ascontiguousarray(W[:, units])
    Qref = c_oracle.quantize_layer(Ws, X, X if Xq is None else Xq, A, nthreads=cores)
    Qg = np.asarray(Qgpu)[:, units]
    agree = float(np.mean(Qref == Qg))
    delta = 0.0
    if agree < 1.0:   # identical Q => identical residual; only mismatching columns can differ
        bad = [i for i in range(len(units)) if not np.array_equal(Qref[:, i], Qg[:, i])]
        r_ref = residual_rel(Ws[:, bad], Qref[:, bad], X, X if Xq is None else Xq)
        r_gpu = residual_rel(Ws[:, bad], Qg[:, bad], X, X if Xq is None else Xq)
        delta = float(np.max(np.abs(r_gpu - r_ref) / np.maximum(r_ref, 1e-300)))
    return {"agreement": agree, "resid_rel_delta": delta, "n_checked": int(Qref.size), "units": len(units)}


# ----------------------------------------------------------------------------------------------------------------
# per-layer roofline
# ----------------------------------------------------------------------------------------------------------------
def layer_roofline(d, sts, ms, hbm_peak, i8_peak):
    """Fraction of the governing roofline of one layer from the library's stage times (gpfq_query_stats) of its call(s)."""
    st = sts[0]
    rec = {"ms": round(ms, 4), "weights_per_s": round(layer_weights(d) / (ms * 1e-3)) if ms > 0 else None}
    if d["kind"] == "conv":
        gk = st.get("gram_kernel")
        ms_g = st["ms_gram"] if st["ms_gram"] > 0 else ms
        rec["form"] = {0: "patch form (shared-memory planes, 126 MACs / column)", 4: "correlation form (13 DFMA / pixel / Gram)",
                       5: "correlation form, packed images"}.get(gk, str(gk))
        hbm = st["bytes_algorithmic"] / (ms_g * 1e-3) / 1e9 / hbm_peak
        pipe = st["flops_algorithmic"] / 2 / (ms_g * 1e-3) / (DFMA_RATE if gk in (4, 5) else DMMA_RATE)
        rec.update(ms_gram=round(ms_g, 4), hbm_frac=round(hbm, 3), fp64_pipe_frac=round(pipe, 3),
                   bound="fp64 pipe (DFMA)" if pipe >= hbm else "hbm", frac=round(max(pipe, hbm), 3))
    else:
        rec["method"] = {1: "stream", 2: "gram", 3: "stream_fast"}.get(st["method"])
        rec["gram_kernel"] = {1: "dmma", 2: "i8_tcgen05", 3: "residual form (block-diagonal tiles)"}.get(st.get("gram_kernel"))
        rec.update(ms_gram=round(st["ms_gram"], 4), ms_sweep=round(st["ms_sweep"], 4), ms_stream=round(st["ms_stream"], 4))
        nj, N0, m = d["j1"] - d["j0"], d["N0"], d["m"]
        if st["method"] == 2:
            macs = 3.0 * m * N0 * nj if st.get("gram_kernel") == 3 else float(N0) * N0 * nj
            i8 = st.get("reserved", 0)
            rec["walk"] = "sweep_tc_kernel (tensor-core range walk)" if i8 & 2 else "sweep_pipe_kernel / sweep_tile_kernel"
            if i8 & 1:      # sweep contractions on tcgen05 (int8 slices): reported against the int8 tensor peak
                ops = float(st["flops_algorithmic"])
                rec.update(bound="tensor (int8 slices on tcgen05)", frac=round(ops / (st["ms_sweep"] * 1e-3) / 1e12 / i8_peak, 3),
                           sweep_form="carried residuals, int8-slice contractions" if st.get("gram_kernel") == 3 else "Gram rows")
            else:
                rec.update(bound="fp64 pipe (DMMA)", frac=round(macs / DMMA_RATE / (max(st["ms_sweep"], 1e-6) * 1e-3), 3),
                           sweep_form="carried residuals: 3 m N0 N1 MACs" if st.get("gram_kernel") == 3 else "Gram rows: N0^2 N1 MACs")
            if st.get("gram_kernel") == 2 and st["ms_gram"] > 0:
                tiles = sum((ti >> 1) + 1 for ti in range(-(-N0 // 128)))
                ops = 15 * tiles * 128 * 256 * 2 * (-(-m // 128) * 128) * (1 if d["first"] else 2)
                rec["gram_int8_frac"] = round(ops / (st["ms_gram"] * 1e-3) / 1e12 / i8_peak, 3)
        else:
            rec.update(bound="fp64 pipe (DFMA)", frac=round(3.0 * m * N0 * nj / DFMA_RATE / (max(st["ms_stream"], 1e-6) * 1e-3), 3))
    return rec


def load_traffic(kernel):
    """DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) against algorithmic bytes of `kernel` from the committed
    `ncu --set full` capture of this round (profiles/r2_traffic.json); None when no capture is committed."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json"))).get(kernel)
    except Exception:
        return None


# ----------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gpfq", choices=["gpfq", "reference"])
    ap.add_argument("--workload", default="vgg16", choices=sorted(WORKLOADS))
    ap.add_argument("--n-img", type=int, default=0, help="override the image / sample count (debug only)")
    ap.add_argument("--e2e-steps", type=int, default=1)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline and parity legs")
    ap.add_argument("--profile", action="store_true", help="profiling only: warm-up + timed passes of the value leg, nothing else")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the Q of every layer of the last step as DIR/<layer>.npy (float64; "
                         "a fixed seeded sample of the larger layers, under 64 MB in all).  With N > 1 GPUs the Dense layers "
                         "come from the fp32 all-gather, so compare dumps of runs with the same GPU count")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "gpfq":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl gpfq)")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = WORKLOADS[args.workload]
    layers = wl["layers"]
    n_img = args.n_img or wl["n_img"]
    total_weights = sum(layer_weights(l) for l in layers)
    cores = len(os.sched_getaffinity(0))
    config = {"workload": f"{args.workload}: {wl['desc']}", "samples": n_img or "per layer",
              "alphabet": f"K={int(round(2 ** wl['bits']))} levels, alphabet_scalar={wl['c']}",
              "weights_per_step": total_weights,
              "sharding": f"conv layers over images + all-reduce of the Grams, Dense neurons over {world} rank(s) + all-gather of Q",
              "l2": wl["l2"]}
    metric = "quantized weights/s, full-network GPFQ pass"

    if args.impl == "reference":
        if rank != 0:
            return
        reference_arm(args, wl, layers, n_img, total_weights, cores, config, metric)
        return

    want_cpu = rank == 0 and world == 1 and not args.no_cpu and not args.no_e2e and not args.profile
    pool = CpuPool(cores) if want_cpu else None      # forked before CUDA exists in this process

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the GPFQ hot path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from quantized_neural_networks_b200 import get_engine
    eng = get_engine(local_rank)

    data = build_device_inputs(wl, n_img, rank, world, dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    W_ = max(args.warmup, 3)
    for _ in range(W_):
        for d in data:
            run_layer_device(eng, d, world)
    barrier()
    if args.profile:
        for _ in range(args.steps):
            for d in data:
                run_layer_device(eng, d, world)
        barrier()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, data, world)
        return
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(len(data) + 1)] for _ in range(args.steps)]
    with ClockSampler(local_rank) as clocks:
        barrier()
        for s in range(args.steps):
            ev[s][0].record()
            for i, d in enumerate(data):
                run_layer_device(eng, d, world)
                ev[s][i + 1].record()
        barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, data, world)
    ms = ev[0][0].elapsed_time(ev[-1][-1])
    layer_ms = [float(np.mean([ev[s][i].elapsed_time(ev[s][i + 1]) for s in range(args.steps)])) for i in range(len(data))]
    if world > 1:
        t = torch.tensor([ms] + layer_ms, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, layer_ms = float(t[0].item()), [float(v) for v in t[1:].tolist()]
    ms_per_step = ms / args.steps
    value = total_weights / (ms_per_step * 1e-3)

    # stage times of the LAST step's calls (most recent call first)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    i8_peak = 2.0 * float(peaks.get("bf16_tflops", 1590.0))
    back, launches_per_step, per_layer, stage = 0, 0, {}, {}
    for i in range(len(data) - 1, -1, -1):
        d = data[i]
        sts = []
        for _ in range(api_calls(d, world)):
            sts.append(eng.query_stats(back))
            back += 1
        sts.reverse()
        launches_per_step += sum(s["kernel_launches"] for s in sts)
        stage[d["name"]] = sts
        per_layer[d["name"]] = layer_roofline(d, sts, layer_ms[i], hbm_peak, i8_peak)
    per_layer = {d["name"]: per_layer[d["name"]] for d in data}

    # the dominant kernel family of the step
    conv_ms = sum(stage[d["name"]][0]["ms_gram"] for d in data if d["kind"] == "conv" and stage[d["name"]][0].get("gram_kernel") in (4, 5))
    conv_bytes = sum(stage[d["name"]][0]["bytes_algorithmic"] for d in data if d["kind"] == "conv" and stage[d["name"]][0].get("gram_kernel") in (4, 5))
    conv_dfma = sum(stage[d["name"]][0]["flops_algorithmic"] / 2 for d in data if d["kind"] == "conv" and stage[d["name"]][0].get("gram_kernel") in (4, 5))
    roofline = None
    traffic = load_traffic("conv_corr9_tma_kernel")
    if conv_ms > 0:
        ach = conv_bytes / (conv_ms * 1e-3) / 1e9
        roofline = {"kernel": "conv_corr9_tma_kernel / conv_corr9_strip_kernel (3x3 per-channel Grams as 13 displacement sums straight from "
                              "the NHWC activations: TMA 4-D boxes -> per-warp mbarrier ring -> fp64 register window, DFMA; bands of "
                              "5-column boxes on 224 / 112-pixel images, whole strips of <= 16 columns as straight-line code below)",
                    "share_of_step": round(conv_ms / ms_per_step, 3), "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                    "frac": ach / hbm_peak,
                    "traffic": None if traffic is None else traffic["ratio"] * conv_bytes,
                    "traffic_note": None if traffic is None else
                    f"DRAM bytes of the same launches = {traffic['ratio']:.3f} x their algorithmic bytes, the ratio ncu measured on "
                    f"{traffic['layer']}: {traffic['note']} ({traffic['capture']})",
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs (copy)" if peaks else "fallback (B200_PROFILING.md)",
                    "algorithmic_bytes": "4 B per pixel and channel per tensor (X and Xq activations, each read once) over the CUDA-event "
                                         "time of the Gram stage of every conv call of the last step",
                    "dfma_pipe_frac": conv_dfma / (conv_ms * 1e-3) / DFMA_RATE,
                    "dfma_pipe_note": "the kernel issues 13 DFMA per pixel, channel and Gram; the fp64 pipe (17.05e12 DFMA/s measured, "
                                      "profiles/fp64_pipes_r1.txt) saturates before HBM does"}

    # ---- e2e + parity + cpu baseline: host (pinned) buffers through the C ABI, layer by layer ----------------------
    e2e, parity, cpu = None, None, None
    if not args.no_e2e:
        e2e, parity, cpu = e2e_leg(args, eng, data, rank, world, dev, pool, cores, total_weights, barrier)
    if pool is not None:
        pool.close()

    if rank == 0:
        line = {"metric": metric, "value": value, "unit": "weights/s", "n_gpus": world, "steps": args.steps, "warmup": W_,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": config, "clocks": clocks.summary(), "e2e": e2e,
                "gpu_launches": int(launches_per_step * args.steps), "roofline": roofline, "parity": parity, "cpu_baseline": cpu,
                "per_layer": per_layer}
        print(json.dumps(line))
        if parity is not None:
            bad = {k: v for k, v in parity.items() if v["agreement"] < 0.9999 or v["resid_rel_delta"] > 1e-6}
            if bad:
                raise SystemExit(f"parity gate failed: {bad}")
    if world > 1:
        dist.destroy_process_group()


def e2e_leg(args, eng, data, rank, world, dev, pool, cores, total_weights, barrier):
    """The pass from HOST buffers.  One pinned buffer pair, refilled per layer from the device tensors OUTSIDE the timed
    region (the reference's host code holds one layer's activations at a time too: layer{idx}_data.h5 is written, used and
    removed per layer, quantized_network.py:471-500, :574); the timed region of a layer is the synchronous C-ABI call(s):
    H2D copies, kernels, D2H of Q.  world > 1: every rank hands over only its own images (conv: image split, one all-reduce
    of the Grams) / samples or a 1 / world slice of the replicated inputs (Dense), see replicate.py."""
    import torch
    import torch.distributed as dist
    from quantized_neural_networks_b200.replicate import prefer_sample_split, replicate_leading_axis, sample_split_gram
    need = max((d["act"].numel() if d["kind"] == "conv" else d["X"].numel()) for d in data)
    pin = [torch.empty(need, dtype=torch.float32, pin_memory=True) for _ in range(2)]

    def host_view(t, which):
        h = pin[which][:t.numel()].view(t.shape)
        h.copy_(t)
        return h.numpy()

    parity = {} if pool is not None else None
    cpu_s, cpu_w, cpu_desc = 0.0, 0, []
    total_s, h2d, d2h = 0.0, 0, 0
    for it in range(1 + args.e2e_steps):      # pass 0: warm-up (allocates the staging workspaces) + parity + CPU sample
        timed = it > 0
        for d in data:
            convl = d["kind"] == "conv"
            a = host_view(d["act"] if convl else d["X"], 0)
            src_q = d["actq"] if convl else d["Xq"]
            aq = None if src_q is None else host_view(src_q, 1)
            Wh = d["W"].cpu().numpy()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            if convl and world == 1:
                Q = eng.conv_layer_nhwc(a, aq, Wh, d["A"])
                nb = a.nbytes * (1 if aq is None else 2)
            elif convl:
                gram = eng.conv_gram_nhwc(a, aq, (3, 3))
                dist.all_reduce(gram)
                Q = eng.conv_layer_from_gram(gram, Wh, d["A"])
                nb = a.nbytes * (1 if aq is None else 2)
            elif world == 1:
                Q = eng.dense_layer(a, aq, Wh, d["A"])
                nb = a.nbytes * (1 if aq is None else 2)
            elif prefer_sample_split(d["N0"], d["m"], world):
                G1, G2 = sample_split_gram(eng, a, aq, rank, world, device=dev)
                Q = eng.dense_layer_from_gram(G1, G2, Wh, d["A"], j0=d["j0"], j1=d["j1"])
                lo, hi = shard_range(d["m"], rank, world)
                nb = d["N0"] * (hi - lo) * 4 * (1 if aq is None else 2)
            else:
                ad = replicate_leading_axis(a, rank, world, dev)
                aqd = None if aq is None else replicate_leading_axis(aq, rank, world, dev)
                Wd = torch.from_numpy(Wh).to(dev, non_blocking=True)
                Q = eng.dense_layer(ad, aqd, Wd, d["A"], j0=d["j0"], j1=d["j1"])[..., d["j0"]:d["j1"]].cpu().numpy()
                nb = -(-d["N0"] // world) * d["m"] * 4 * (1 if aq is None else 2)
                del ad, aqd
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if timed:
                total_s += dt
                if it == 1:
                    h2d += nb + Wh.nbytes
                    d2h += (layer_weights(d) if world == 1 or convl else d["N0"] * (d["j1"] - d["j0"])) * 8
            elif pool is not None:
                # ---- parity at full size on the host buffers just handed to the C ABI, and the CPU-baseline sample
                Q0 = Q
                if convl:
                    c = d["C"] // 2
                    plane = np.ascontiguousarray(a[..., c])
                    planeq = None if aq is None else np.ascontiguousarray(aq[..., c])
                    Xp = plane_patches(plane)
                    Xqp = None if planeq is None else plane_patches(planeq)
                    units = range(min(d["F"], 16 if Xp.shape[1] > 10_000_000 else 32))
                    parity[d["name"]] = parity_layer(d, Wh[:, :, c, :].reshape(9, -1), d["A"], Q0[:, :, c, :].reshape(9, -1), Xp, Xqp, units, cores)
                    del Xp, Xqp
                    sec, w, desc = cpu_time_layer(pool, dict(d, n_img_total=d["n_img"]), Wh[:, :, c, :], d["A"], planes=(plane, planeq))
                else:
                    units = range(min(d["N1"], 2 * cores if d["N0"] * d["m"] > 3e7 else 4 * cores))
                    parity[d["name"]] = parity_layer(d, Wh, d["A"], Q0, a, aq, units, cores)
                    sec, w, desc = cpu_time_layer(pool, d, Wh, d["A"], X=a, Xq=aq)
                cpu_s += sec
                cpu_w += w
                cpu_desc.append(desc)
            del Q
    if world > 1:
        t = torch.tensor([total_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_s = float(t.item())
    e2e = {"value": total_weights * args.e2e_steps / total_s, "unit": "weights/s", "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": int(d2h), "steps": args.e2e_steps, "ms_per_step": total_s / args.e2e_steps * 1e3,
           "timing": "host wall clock around the synchronous C-ABI call(s) of every layer (H2D copies + kernels + D2H of Q), "
                     "summed over the layers, max over ranks; the pinned host buffers are refilled between layers outside the timed region",
           "api": ("gpfq_conv_layer_nhwc + gpfq_dense_layer from pinned host buffers" if world == 1 else
                   f"per rank 1/{world} of every input over PCIe: gpfq_conv_gram_nhwc on the rank's images + all-reduce + "
                   "gpfq_conv_layer_from_gram; Dense: sample split (gpfq_gram_matrices + all-reduce + gpfq_dense_layer_from_gram) when "
                   "m > 2 N0, else inputs replicated by one all-gather over NVLink (bytes are per rank)")}
    cpu = None
    if pool is not None:
        cpu = {"value": total_weights / cpu_s, "unit": "weights/s", "cores": cores, "kind": "port",
               "sample": "NumPy port of the reference walk, one process per core; per layer [filters or neurons timed / total x images "
                         "used / total]: " + " ".join(cpu_desc) + "; extrapolated linearly; HDF5 I/O excluded",
               "sampled_weights": int(cpu_w), "extrapolated_full_pass_s": cpu_s}
    return e2e, parity, cpu


def reference_arm(args, wl, layers, n_img, total_weights, cores, config, metric):
    """The reference's own CPU implementation of the path: Python / NumPy, does not travel to the GPU box -> the oracle's
    NumPy port, run exactly as BASELINE.md section 3 prescribes (one process per core, single-threaded BLAS).  A step is a
    bounded sample of every layer; `value` extrapolates it linearly to the whole pass, `ms_per_step` is the sample itself."""
    pool = CpuPool(cores)
    rng = np.random.default_rng(0)
    samples = []
    for li, l in enumerate(layers):
        first = li == 0
        if l["kind"] == "conv":
            C, F, H = l["C"], l["F"], l["H"]
            W = (rng.uniform(-1, 1, (3, 3, F)) * np.sqrt(6.0 / (9 * C))).astype(np.float32)   # the filters of ONE channel
            n_s = max(1, min(n_img, 600_000 // (H * H)))
            if first:
                plane = rng.random((n_s, H, H), dtype=np.float32)
                planes = (plane, None)
            else:
                Z = rng.standard_normal((n_s, H, H), dtype=np.float32)
                planes = (np.maximum(Z, 0), np.maximum(Z + 0.05 * rng.standard_normal((n_s, H, H), dtype=np.float32), 0))
            A = make_alphabet(np.median(np.abs(W)), wl)
            samples.append((dict(l, n_img_total=n_img), W, A, dict(planes=planes)))
        else:
            N0, N1 = l["N0"], l["N1"]
            m = l["m"] or n_img
            take = min(N1, 2 * cores if N0 >= 1024 else 4 * cores)
            W = (rng.uniform(-1, 1, (N0, take)) * np.sqrt(6.0 / N0)).astype(np.float32)
            Z = rng.standard_normal((N0, m), dtype=np.float32)
            X = np.maximum(Z, 0)
            Xq = None if first else np.maximum(Z + 0.05 * rng.standard_normal((N0, m), dtype=np.float32), 0)
            del Z
            A = make_alphabet(np.median(np.abs(W)), wl)
            samples.append((dict(l), W, A, dict(X=X, Xq=Xq)))
    vals, walls, desc = [], [], ""
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        sec, descs = 0.0, []
        for l, W, A, kw in samples:
            s, w, dsc = cpu_time_layer(pool, l, W, A, **kw)
            sec += s
            descs.append(dsc)
        if it >= args.warmup:
            vals.append(total_weights / sec)
            walls.append(time.perf_counter() - t0)
        desc = " ".join(descs)
    pool.close()
    v = float(np.mean(vals))
    line = {"impl": "reference", "metric": metric, "value": v, "unit": "weights/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(np.mean(walls)) * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "value_note": "whole-pass weights/s extrapolated linearly from the sample each step walks; ms_per_step is the wall time "
                          "of that sample; extrapolated_full_pass_s the whole pass at this rate",
            "cpu_baseline": {"value": v, "unit": "weights/s", "cores": cores, "kind": "port",
                             "sample": "NumPy port of the reference walk, one process per core; per layer [filters or neurons timed / "
                                       "total x images used / total]: " + desc + "; extrapolated linearly; HDF5 I/O excluded",
                             "extrapolated_full_pass_s": total_weights / v},
            "e2e": {"value": v, "unit": "weights/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
