"""Conv layers with kernels other than 3 x 3 at realistic sizes: median time per layer through the public engine API.

    python tools/conv_kk_bench.py [--mem-gb 12] [--reps 5] [--warmup 1] [--dump DIR] [--only NAME ...]
    python tools/conv_kk_bench.py --compare DIR_A DIR_B

Layers: AlexNet conv1 (11 x 11 / 4 VALID, 3 -> 64, 227 x 227, first-layer form), AlexNet conv2 (5 x 5 SAME, 64 -> 192, 27 x 27),
the ResNet stem (7 x 7 / 2 SAME, 3 -> 64, 224 x 224, first-layer form), Inception-v3 1 x 7 and 7 x 1 (192 -> 192, 17 x 17) and an
Inception 5 x 5 branch (48 -> 64, 35 x 35).  Activations are device-resident and seeded (torch's CUDA generator), with as many
images as fit in --mem-gb for the activations plus the patch matrices of every channel.  Only `conv_layer_nhwc` is timed;
`conv_gram_nhwc` is tried once per layer and reported as `gram_only_path` (builds that lack it for a kernel size raise
GpfqError there), so the same file runs on any build of the library.

Per layer: median ms over --reps synchronised calls after --warmup, and the algorithmic MACs of the two Grams (kk (kk + 1) / 2
per patch column, channel and Gram: lower triangles + diagonals; one Gram in the first-layer form) over that time as a share of
the project's measured DMMA rate (18.55e12 FMA/s, DESIGN.md section 5).  The GPU name and power limit come from the same run.
--dump DIR writes each layer's Q as DIR/<layer>.npy; --compare prints the agreement of two such directories.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

DMMA_FMA = 18.55e12
# name: (kernel, strides, padding, C, F, H (= W), first-layer form)
LAYERS = {
    "alexnet_conv1_11x11s4": ((11, 11), (4, 4), "VALID", 3, 64, 227, True),
    "alexnet_conv2_5x5": ((5, 5), (1, 1), "SAME", 64, 192, 27, False),
    "resnet_stem_7x7s2": ((7, 7), (2, 2), "SAME", 3, 64, 224, True),
    "inception_1x7": ((1, 7), (1, 1), "SAME", 192, 192, 17, False),
    "inception_7x1": ((7, 1), (1, 1), "SAME", 192, 192, 17, False),
    "inception_5x5": ((5, 5), (1, 1), "SAME", 48, 64, 35, False),
}


def out_size(H, k, s, pad):
    return -(-H // s) if pad == "SAME" else (H - k) // s + 1


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def compare(a, b):
    for f in sorted(os.listdir(a)):
        if f.endswith(".npy") and os.path.exists(os.path.join(b, f)):
            qa, qb = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
            print(json.dumps({"layer": f[:-4], "agreement": float(np.mean(qa == qb)), "entries": int(qa.size)}))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--mem-gb", type=float, default=12.0, help="device memory for activations + patch matrices")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--dump", default=None, help="write each layer's Q as DIR/<layer>.npy")
    ap.add_argument("--only", nargs="*", default=None)
    ap.add_argument("--compare", nargs=2, default=None, metavar=("DIR_A", "DIR_B"))
    args = ap.parse_args()
    if args.compare:
        compare(*args.compare)
        return
    import torch
    from quantized_neural_networks_b200 import GpfqError, get_engine
    if not torch.cuda.is_available():
        sys.exit("conv_kk_bench: no CUDA device")
    eng = get_engine(0)
    name, power = gpu_info()
    print(json.dumps({"gpu": name, "power_limit": power}), flush=True)
    if args.dump:
        os.makedirs(args.dump, exist_ok=True)
    for li, (lname, (ks, st, pad, C, F, H, first)) in enumerate(LAYERS.items()):
        if args.only and lname not in args.only:
            continue
        kk = ks[0] * ks[1]
        Ho, Wo = out_size(H, ks[0], st[0], pad), out_size(H, ks[1], st[1], pad)
        mats = 1 if first else 2
        per_img = mats * (H * H * C + kk * Ho * Wo * C) * 4
        n_img = max(1, int(args.mem_gb * 2**30 // per_img))
        g = torch.Generator(device="cuda").manual_seed(1000 + li)
        act = torch.relu(torch.randn((n_img, H, H, C), generator=g, device="cuda"))
        actq = None if first else torch.relu(act + 0.05 * torch.randn(act.shape, generator=g, device="cuda"))
        fan = kk * C
        W = ((torch.rand((*ks, C, F), generator=g, device="cuda") * 2 - 1) * np.sqrt(6.0 / (fan + kk * F))).contiguous()
        A = 2 * float(W.abs().median()) * np.linspace(-1, 1, 3)
        geo = dict(strides=st, padding=pad)
        try:   # builds without a Gram-only path for this kernel size raise here; the timed call still runs
            eng.conv_gram_nhwc(act[:1], None if first else actq[:1], ks, **geo)
            gram_only = True
        except GpfqError:
            gram_only = False
        for _ in range(args.warmup):
            Q = eng.conv_layer_nhwc(act, actq, W, A, **geo)
        times = []
        for _ in range(args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            Q = eng.conv_layer_nhwc(act, actq, W, A, **geo)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        ms = float(np.median(times)) * 1e3
        n = n_img * Ho * Wo
        macs = (1 if first else 2) * kk * (kk + 1) // 2 * n * C
        print(json.dumps({"layer": lname, "kk": kk, "C": C, "F": F, "n_img": n_img, "patches_per_channel": n,
                          "median_ms": round(ms, 3), "min_ms": round(min(times) * 1e3, 3), "gram_macs": macs,
                          "dmma_share": round(macs / (ms * 1e-3) / DMMA_FMA, 4),
                          "kernel_launches": eng.last_stats.get("kernel_launches"), "gram_only_path": gram_only}), flush=True)
        if args.dump:
            np.save(os.path.join(args.dump, lname + ".npy"), Q.cpu().numpy())
        del act, actq, W, Q
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
