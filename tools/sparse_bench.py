"""Sparse GPFQ: the call without the L1 penalty against the call with it, at realistic sizes, through the public engine API.

    python tools/sparse_bench.py [--reps 3] [--warmup 1] [--only NAME ...]

Layers (hidden-layer form, X != Xq, seeded device-resident inputs, ternary per-layer alphabets), those of
tools/channel_alphabet_bench.py:
  * vgg16_fc1        Dense 25088 -> 4096, m = 1504 (residual form of the sweep)
  * vgg16_fc2        Dense 4096 -> 4096, m = 1504
  * dense_4096_25k   Dense 4096 -> 4096, m = 25000 (Gram rows)
  * cifar_conv2      Conv2D 3 x 3, 32 -> 32 channels, 32 x 32 images, 5008 images
  * dw3x3_14_512     DepthwiseConv2D 3 x 3 on 14 x 14 x 512 (groups = C), 1504 images
  * convnext_t_dw7   ConvNeXt-T stage-1 depthwise 7 x 7 on 56 x 56 x 96, 256 images
Per layer: median ms over --reps synchronised calls after --warmup of the call without the penalty and of the calls with the lambdas
that zero about 30 % and about 70 % of the weights (found by bisection on lambda = c * a * median ||Xq_t||^2), each lambda's zero
fraction and relative residual ||X^T W - Xq^T Q|| / ||X^T W|| (the layer outputs before the bias), the kernels each ran
(`gram_kernel`, `reserved`: bit 0 int8 residual form, bit 1 tensor-core walk; every call runs the same kernels) and the
penalty / no-penalty time ratios.  The GPU name and power limit come from the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# name: ("dense", N0, N1, m) | ("conv", kernel, C, F, groups, H, n_img)
LAYERS = {
    "vgg16_fc1": ("dense", 25088, 4096, 1504),
    "vgg16_fc2": ("dense", 4096, 4096, 1504),
    "dense_4096_25k": ("dense", 4096, 4096, 25000),
    "cifar_conv2": ("conv", (3, 3), 32, 32, 1, 32, 5008),
    "dw3x3_14_512": ("conv", (3, 3), 512, 512, 512, 14, 1504),
    "convnext_t_dw7": ("conv", (7, 7), 96, 96, 96, 56, 256),
}


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def timed(fn, reps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return float(np.median(times)) * 1e3


def calibrate(run, target, lo=1e-4, hi=1e2, iters=12):
    """c with zero fraction of run(c) ~ target (bisection in log c; the fraction grows with c)."""
    for _ in range(iters):
        mid = float(np.sqrt(lo * hi))
        if run(mid) < target:
            lo = mid
        else:
            hi = mid
    return float(np.sqrt(lo * hi))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", nargs="*", default=None)
    args = ap.parse_args()
    import torch
    import torch.nn.functional as tf
    from quantized_neural_networks_b200 import get_engine
    if not torch.cuda.is_available():
        sys.exit("sparse_bench: no CUDA device")
    eng = get_engine(0)
    name, power = gpu_info()
    print(json.dumps({"gpu": name, "power_limit": power}), flush=True)
    base = np.linspace(-1, 1, 3)
    for li, (lname, spec) in enumerate(LAYERS.items()):
        if args.only and lname not in args.only:
            continue
        g = torch.Generator(device="cuda").manual_seed(3000 + li)
        if spec[0] == "dense":
            _, N0, N1, m = spec
            X = torch.relu(torch.randn((N0, m), generator=g, device="cuda"))
            Xq = torch.relu(X + 0.05 * torch.randn((N0, m), generator=g, device="cuda"))
            W = ((torch.rand((N0, N1), generator=g, device="cuda") * 2 - 1) * np.sqrt(6.0 / (N0 + N1))).contiguous()
            A = np.float32(3) * np.median(np.abs(W.cpu().numpy().flatten())) * base
            den = float(torch.median((Xq.double() ** 2).sum(1)))
            call = lambda lam=None, j1=None: eng.dense_layer(X, Xq, W, A, j1=j1, **({} if lam is None else {"l1_penalty": lam}))
            part = lambda lam: call(lam, j1=min(N1, 256))[:, :min(N1, 256)]
            ref = (X.double().T @ W.double())
            resid = lambda Q: float(torch.linalg.norm(ref - Xq.double().T @ Q) / torch.linalg.norm(ref))
            shape = {"N0": N0, "N1": N1, "m": m}
        else:
            _, ks, C, F, groups, H, n_img = spec
            act = torch.relu(torch.randn((n_img, H, H, C), generator=g, device="cuda"))
            actq = torch.relu(act + 0.05 * torch.randn(act.shape, generator=g, device="cuda"))
            Cg = C // groups
            W = ((torch.rand((*ks, Cg, F), generator=g, device="cuda") * 2 - 1) * 0.2).contiguous()
            A = np.float32(3) * np.median(np.abs(W.cpu().numpy().flatten())) * base
            gk = {"groups": groups} if groups > 1 else {}
            den = float(torch.median((actq.double() ** 2).sum((0, 1, 2))))   # ~ ||Xq_t||^2 of a tap's patch row
            call = lambda lam=None: eng.conv_layer_nhwc(act, actq, W, A, **gk, **({} if lam is None else {"l1_penalty": lam}))
            part = call
            nchw = lambda a: a.permute(0, 3, 1, 2).double()
            conv = lambda a, k: tf.conv2d(nchw(a), k.permute(3, 2, 0, 1).double(), padding="same", groups=groups)
            ref = conv(act, W)
            resid = lambda Q: float(torch.linalg.norm(ref - conv(actq, Q)) / torch.linalg.norm(ref))
            shape = {"kernel": list(ks), "C": C, "F": F, "groups": groups, "H": H, "n_img": n_img}
        scale = float(A[-1]) * den
        zf = lambda Q: float((Q == 0).double().mean()) if torch.is_tensor(Q) else float(np.mean(Q == 0))
        ms_off = timed(lambda: call(), args.reps, args.warmup)
        st_off = dict(eng.last_stats)
        Q_off = call()
        row = {"layer": lname, **shape, "off_ms": round(ms_off, 3), "off_zero_fraction": round(zf(Q_off), 4),
               "off_residual": round(resid(Q_off), 5), "gram_kernel": [st_off["gram_kernel"]], "reserved": [st_off["reserved"]]}
        for target in (0.3, 0.7):
            c = calibrate(lambda cc: zf(part(cc * scale)), target)
            lam = c * scale
            ms = timed(lambda: call(lam), args.reps, args.warmup)
            st = dict(eng.last_stats)
            Q = call(lam)
            tag = f"l1_{int(target * 100)}"
            row.update({f"{tag}_lambda": lam, f"{tag}_ms": round(ms, 3), f"{tag}_zero_fraction": round(zf(Q), 4),
                        f"{tag}_residual": round(resid(Q), 5), f"{tag}_ratio": round(ms / ms_off, 3)})
            row["gram_kernel"].append(st["gram_kernel"])
            row["reserved"].append(st["reserved"])
        print(json.dumps(row), flush=True)
        del W
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
