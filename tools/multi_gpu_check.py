"""Multi-GPU check, run under torchrun (one rank per GPU, NCCL):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/multi_gpu_check.py

Every rank quantizes an MNIST-shaped MLP through the mirror API three ways -- unsharded on its own GPU, sharded with the
layer inputs replicated (1 / world over PCIe + NVLink all-gather), and sharded with the Gram stage split over samples
(partial Grams + NCCL all-reduce, `gpfq_dense_layer_from_gram`) -- and compares the quantized kernels and the predictions.
Replication must be bit-identical to the one-GPU pass; the sample split re-associates fp64 sums, so the north-star gate
applies (>= 99.99 % of entries, identical predictions).  Also times the two Dense feeds on a config-4-like layer.
Prints `MULTI_GPU_CHECK PASS` from rank 0 when every rank agrees."""
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from quantized_neural_networks_b200 import QuantizedCNN, QuantizedNeuralNetwork, get_engine, hostnet  # noqa: E402
from quantized_neural_networks_b200.replicate import replicate_leading_axis, sample_split_gram, shard_range  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ok = True
    log = (lambda *a: print(*a, flush=True)) if rank == 0 else (lambda *a: None)

    # ---- full network through the mirror classes -------------------------------------------------------
    rng = np.random.default_rng(0)
    n_img = 2400
    x = (rng.random((n_img, 28, 28)) * (rng.random((n_img, 28, 28)) < 0.5)).astype(np.float32)
    y = rng.integers(0, 10, n_img)
    x_eval = rng.random((512, 28, 28)).astype(np.float32)
    quiet = type("L", (), {"info": staticmethod(lambda m: None)})()

    def run(**kw):
        net = hostnet.mnist_mlp(seed=3, widths=(500, 300), n_in=784, n_out=10)
        q = QuantizedNeuralNetwork(net, 32, hostnet.ArraySequence(x, y, 32), logger=quiet, bits=np.log2(3),
                                   alphabet_scalar=2, device=local, **kw)
        q.quantize_network()
        return q

    one = run()
    rep = run(shard=(rank, world), gram_split="replicate")
    spl = run(shard=(rank, world), gram_split="samples")
    auto = run(shard=(rank, world))
    p_one = one.quantized_net.predict(x_eval).argmax(-1)
    for name, q, exact in (("replicate", rep, True), ("samples", spl, False), ("auto", auto, False)):
        for idx in one.layer_dims:
            a = one.quantized_net.layers[idx].get_weights()[0]
            b = q.quantized_net.layers[idx].get_weights()[0]
            agree = float(np.mean(a == b))
            good = agree == 1.0 if exact else agree >= 0.9999
            ok = ok and good
            log(f"[{name}] layer {idx} {a.shape}: agreement with the one-GPU pass {agree:.6f} {'ok' if good else 'FAIL'}"
                f" (gram_kernel {q.layer_stats[idx].get('gram_kernel')})")
        same_pred = bool(np.array_equal(p_one, q.quantized_net.predict(x_eval).argmax(-1)))
        ok = ok and same_pred
        log(f"[{name}] predictions identical: {same_pred}")
    # the split really ran: the sweep-only entry point reports no Gram kernel of its own
    ok = ok and all(spl.layer_stats[i]["gram_kernel"] == 0 for i in spl.layer_dims)
    ok = ok and auto.layer_stats[1]["gram_kernel"] == 0          # 784 x 2400: m > 2 N0 -> split

    # ---- a CNN: conv layers split over images (per-channel Grams + one tiny all-reduce), Dense layers as above -----------
    xi = rng.random((320, 16, 16, 3)).astype(np.float32)
    xi_eval = rng.random((256, 16, 16, 3)).astype(np.float32)

    def run_cnn(**kw):
        # after the first conv a 5 x 5 layer (image split, like the 3 x 3 layers), a 13 x 11 layer (kernels above 128 taps have
        # no Gram-only path and leave the image split for channel shards) and a grouped 3 x 3 (groups 8: image split with the
        # grouped walk; with gram_split="replicate", ranks take whole groups and gather their filters)
        base = hostnet.cifar10_cnn(seed=5, size=16, widths=(32, 32, 64), dense=64, n_out=10).layers
        net = hostnet.Sequential(base[:2] + [hostnet.Conv2D(32, 5, padding="same", activation="relu"),
                                             hostnet.Conv2D(32, (13, 11), padding="same", activation="relu"),
                                             hostnet.Conv2D(32, 3, padding="same", groups=8, activation="relu")] + base[2:],
                                 input_shape=(16, 16, 3), seed=5)
        q = QuantizedCNN(net, 32, hostnet.ArraySequence(xi, np.zeros(320), 32), logger=quiet, bits=2, alphabet_scalar=3,
                         device=local, **kw)
        q.quantize_network()
        return q

    c_one = run_cnn()
    c_img = run_cnn(shard=(rank, world))
    c_rep = run_cnn(shard=(rank, world), gram_split="replicate")
    pc = c_one.quantized_net.predict(xi_eval).argmax(-1)
    for name, q, exact in (("image split", c_img, False), ("replicate", c_rep, True)):
        for idx, layer in enumerate(c_one.trained_net.layers):
            if layer.__class__.__name__ not in ("Conv2D", "Dense"):
                continue
            a = c_one.quantized_net.layers[idx].get_weights()[0]
            b = q.quantized_net.layers[idx].get_weights()[0]
            agree = float(np.mean(a == b))
            good = agree == 1.0 if exact else agree >= 0.9999
            ok = ok and good
            log(f"[cnn {name}] layer {idx} {layer.__class__.__name__} {a.shape}: agreement {agree:.6f} {'ok' if good else 'FAIL'}")
        same_pred = bool(np.array_equal(pc, q.quantized_net.predict(xi_eval).argmax(-1)))
        ok = ok and same_pred
        log(f"[cnn {name}] predictions identical: {same_pred}")

    # ---- timing of the two feeds on one larger layer (host inputs, all transfers inside) -------------------
    N0, N1, m = 2048, 2048, 40000
    Z = rng.standard_normal((N0, m)).astype(np.float32)
    X = np.maximum(Z, 0)
    Xq = np.maximum(Z + 0.05 * rng.standard_normal((N0, m)).astype(np.float32), 0)
    W = (rng.uniform(-1, 1, (N0, N1)) * np.sqrt(6.0 / (N0 + N1))).astype(np.float32)
    A = 2 * np.median(np.abs(W)) * np.linspace(-1, 1, 3)
    eng = get_engine(local)
    lo, hi = shard_range(N1, rank, world)
    Wd = torch.from_numpy(W).to(dev)
    res = {}
    for mode in ("replicate", "samples", "replicate", "samples"):
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if mode == "replicate":
            Xd = replicate_leading_axis(X, rank, world, dev)
            Xqd = replicate_leading_axis(Xq, rank, world, dev)
            Q = eng.dense_layer(Xd, Xqd, Wd, A, j0=lo, j1=hi, method="gram")
        else:
            G1, G2 = sample_split_gram(eng, X, Xq, rank, world, device=dev)
            Q = eng.dense_layer_from_gram(G1, G2, Wd, A, j0=lo, j1=hi)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device=dev)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        res[mode] = (float(dt[0]) * 1e3, Q[:, lo:hi].clone())
    agree = float((res["replicate"][1] == res["samples"][1]).double().mean())
    ok = ok and agree >= 0.9999
    log(f"Dense ({N0}, {N1}, m={m}) on {world} GPUs from host arrays: replicate {res['replicate'][0]:.1f} ms, "
        f"sample split {res['samples'][0]:.1f} ms (max over ranks, second pass); Q agreement {agree:.6f}")

    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("MULTI_GPU_CHECK " + ("PASS" if int(flag[0]) == 1 else "FAIL"), flush=True)
    dist.destroy_process_group()
    sys.exit(0 if int(flag[0]) == 1 else 1)


if __name__ == "__main__":
    main()
