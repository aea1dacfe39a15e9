"""Grouped Conv2D layers at realistic sizes: one grouped call against `groups` ungrouped calls, through the public engine API.

    python tools/grouped_conv_bench.py [--mem-gb 8] [--reps 5] [--warmup 1] [--only NAME ...]

Layers: a ResNeXt-50 conv2 3 x 3 (128 -> 128, groups 32, 56 x 56), a RegNetX-200MF stage-2 3 x 3 (56 -> 56, group width 8,
28 x 28), the ConvNeXt-T stage-1 depthwise 7 x 7 written as Conv2D(groups=96) (96 -> 96, 56 x 56) and a ShuffleNet 1 x 1 (240 ->
240, groups 3, 28 x 28), all in the hidden-layer form (X != Xq).  Activations are device-resident and seeded (torch's CUDA
generator), with as many images as fit in --mem-gb for the two activation tensors and the patch matrices of every channel.

Per layer: median ms over --reps synchronised calls after --warmup of
  * grouped    one `conv_layer_nhwc(..., groups=groups)` call on the whole layer;
  * per_group  `groups` ungrouped `conv_layer_nhwc` calls, one per group, each on its own contiguous channel slice of the
               activations and its own filter slice of the kernel (the slices are made once, outside the timed window);
and whether the two give the same Q (`q_agreement`: share of equal entries; the per-group calls sum the Gram partials of fewer
channels per launch, so their column chunks, and with them the fp64 summation order, may differ).  The GPU name and power
limit come from the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# name: (kernel, strides, padding, C, F, groups, H (= W))
LAYERS = {
    "resnext50_conv2_3x3_g32": ((3, 3), (1, 1), "SAME", 128, 128, 32, 56),
    "regnetx200mf_s2_3x3_gw8": ((3, 3), (1, 1), "SAME", 56, 56, 7, 28),
    "convnext_t_s1_7x7_g96": ((7, 7), (1, 1), "SAME", 96, 96, 96, 56),
    "shufflenet_1x1_g3": ((1, 1), (1, 1), "SAME", 240, 240, 3, 28),
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


def timed(fn, reps, warmup):
    import torch
    for _ in range(warmup):
        out = fn()
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return out, times


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--mem-gb", type=float, default=8.0, help="device memory for the activations + patch matrices")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", nargs="*", default=None)
    args = ap.parse_args()
    import torch
    from quantized_neural_networks_b200 import get_engine
    if not torch.cuda.is_available():
        sys.exit("grouped_conv_bench: no CUDA device")
    eng = get_engine(0)
    name, power = gpu_info()
    print(json.dumps({"gpu": name, "power_limit": power}), flush=True)
    for li, (lname, (ks, st, pad, C, F, groups, H)) in enumerate(LAYERS.items()):
        if args.only and lname not in args.only:
            continue
        kk = ks[0] * ks[1]
        Cg, Fg = C // groups, F // groups
        Ho, Wo = out_size(H, ks[0], st[0], pad), out_size(H, ks[1], st[1], pad)
        per_img = 2 * (2 * H * H * C + kk * Ho * Wo * C) * 4      # activations twice (whole + group slices), patches
        n_img = max(1, int(args.mem_gb * 2**30 // per_img))
        g = torch.Generator(device="cuda").manual_seed(2000 + li)
        act = torch.relu(torch.randn((n_img, H, H, C), generator=g, device="cuda"))
        actq = torch.relu(act + 0.05 * torch.randn(act.shape, generator=g, device="cuda"))
        W = ((torch.rand((*ks, Cg, F), generator=g, device="cuda") * 2 - 1) * np.sqrt(6.0 / (kk * Cg + kk * Fg))).contiguous()
        A = 2 * float(W.abs().median()) * np.linspace(-1, 1, 3)
        geo = dict(strides=st, padding=pad)

        Qg, tg = timed(lambda: eng.conv_layer_nhwc(act, actq, W, A, groups=groups, **geo), args.reps, args.warmup)
        launches = eng.last_stats.get("kernel_launches")
        slices = [(act[..., i * Cg:(i + 1) * Cg].contiguous(), actq[..., i * Cg:(i + 1) * Cg].contiguous(),
                   W[..., i * Fg:(i + 1) * Fg].contiguous()) for i in range(groups)]

        def per_group():
            return [eng.conv_layer_nhwc(a, aq, w, A, **geo) for a, aq, w in slices]
        Qs, tp = timed(per_group, args.reps, args.warmup)
        Qp = torch.cat(Qs, dim=3)
        agree = float((Qg == Qp).double().mean())
        ms_g, ms_p = float(np.median(tg)) * 1e3, float(np.median(tp)) * 1e3
        print(json.dumps({"layer": lname, "kk": kk, "C": C, "F": F, "groups": groups, "n_img": n_img,
                          "patches_per_channel": n_img * Ho * Wo, "grouped_ms": round(ms_g, 3), "per_group_ms": round(ms_p, 3),
                          "speedup": round(ms_p / ms_g, 2), "grouped_launches": launches, "q_agreement": agree}), flush=True)
        del act, actq, W, Qg, Qs, Qp, slices
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
