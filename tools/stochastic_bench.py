"""Nearest against stochastic rounding (SPFQ) at realistic sizes, through the public engine API.

    python tools/stochastic_bench.py [--reps 3] [--warmup 1] [--only NAME ...]

Layers (hidden-layer form, X != Xq, seeded device-resident inputs, ternary per-layer alphabets), those of
tools/channel_alphabet_bench.py:
  * vgg16_fc1        Dense 25088 -> 4096, m = 1504 (residual form of the sweep)
  * vgg16_fc2        Dense 4096 -> 4096, m = 1504
  * dense_4096_25k   Dense 4096 -> 4096, m = 25000 (Gram rows)
  * cifar_conv2      Conv2D 3 x 3, 32 -> 32 channels, 32 x 32 images, 5008 images
  * dw3x3_14_512     DepthwiseConv2D 3 x 3 on 14 x 14 x 512 (groups = C), 1504 images
  * convnext_t_dw7   ConvNeXt-T stage-1 depthwise 7 x 7 on 56 x 56 x 96, 256 images
Per layer: median ms over --reps synchronised calls after --warmup of the nearest call and of the stochastic call (one seed), the
kernels each ran (`gram_kernel`, `reserved`: bit 0 int8 residual form, bit 1 tensor-core walk; both calls run the same kernels)
and the stochastic / nearest time ratio.  The GPU name and power limit come from the same run.
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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", nargs="*", default=None)
    args = ap.parse_args()
    import torch
    from quantized_neural_networks_b200 import get_engine
    if not torch.cuda.is_available():
        sys.exit("stochastic_bench: no CUDA device")
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
            Wh = W.cpu().numpy()
            A = np.float32(3) * np.median(np.abs(Wh.flatten())) * base
            nearest_sall = lambda: eng.dense_layer(X, Xq, W, A)
            stoch_call = lambda: eng.dense_layer(X, Xq, W, A, seeds=12345)
            shape = {"N0": N0, "N1": N1, "m": m}
        else:
            _, ks, C, F, groups, H, n_img = spec
            act = torch.relu(torch.randn((n_img, H, H, C), generator=g, device="cuda"))
            actq = torch.relu(act + 0.05 * torch.randn(act.shape, generator=g, device="cuda"))
            Cg = C // groups
            W = ((torch.rand((*ks, Cg, F), generator=g, device="cuda") * 2 - 1) * 0.2).contiguous()
            Wh = W.cpu().numpy()
            A = np.float32(3) * np.median(np.abs(Wh.flatten())) * base
            gk = {"groups": groups} if groups > 1 else {}
            nearest_sall = lambda: eng.conv_layer_nhwc(act, actq, W, A, **gk)
            stoch_call = lambda: eng.conv_layer_nhwc(act, actq, W, A, seeds=12345, **gk)
            shape = {"kernel": list(ks), "C": C, "F": F, "groups": groups, "H": H, "n_img": n_img}
        ms_n = timed(nearest_sall, args.reps, args.warmup)
        st_n = dict(eng.last_stats)
        ms_s = timed(stoch_call, args.reps, args.warmup)
        st_s = dict(eng.last_stats)
        print(json.dumps({"layer": lname, **shape, "nearest_ms": round(ms_n, 3), "stochastic_ms": round(ms_s, 3),
                          "ratio": round(ms_s / ms_n, 3), "gram_kernel": [st_n["gram_kernel"], st_s["gram_kernel"]],
                          "reserved": [st_n["reserved"], st_s["reserved"]]}), flush=True)
        del W
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
