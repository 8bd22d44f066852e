#!/usr/bin/env python
"""Device-timed cost of the clustered RNN (RNNCluster) on one GPU.

    python tools/bench_cluster.py [--steps 10] [--warmup 3] [--out bench_cluster.json]

1. ms per training step of RNNCluster against RNNSampling on the C3 shape (LSTM 2x256, 50k items, max_length 200,
   batch 512, S = 32, Blackout, cluster type mix), with C = 10 and C = 100 clusters.  Both models run the same
   batches; the step is timed with CUDA events around `--steps` steps after `--warmup` untimed ones, and the models
   are measured in alternating rounds.
2. sbr_cluster_topk against sbr_topk (full catalog) at 500k items, H = 512, 256 rows, with C = 10, 50 and 200.  R is
   a planted partition (each item positive in exactly one cluster), so a row scores about N / C items.  A random R
   (0.1 randn, the training initialisation) puts every item in about half of the clusters: it gives no reduction,
   and one such run at C = 50 is reported to show it.

Prints one JSON document and writes it to --out, with the GPU name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from sbr_b200 import _capi  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power, clock = [x.strip() for x in out[0].split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:      # the numbers below stay valid; say where the description is missing
        return dict(gpu="unknown (%s)" % e)


def batches(rng, n, B, T, N, lo=100):
    out = []
    for _ in range(n):
        lens = rng.randint(lo, T + 1, B)
        X = np.zeros((B, T, 1), np.int32)
        mask = np.zeros((B, T), np.float32)
        for b in range(B):
            X[b, :lens[b], 0] = rng.randint(0, N, lens[b])
            mask[b, :lens[b]] = 1
        out.append((X, mask, rng.randint(0, N, B).astype(np.int32)))
    return out


def train_steps(args):
    N, T, B, S = 50000, 200, 512, 32
    rng = np.random.RandomState(0)
    data = batches(rng, 4, B, T, N)
    samples = [rng.randint(0, N, S).astype(np.int32) for _ in range(8)]
    common = dict(n_items=N, cell="LSTM", layers=(256, 256), max_length=T, batch_size=B, n_samples=S, updater="adam")
    models = {"sampling": _capi.Engine(loss="Blackout", **common)}
    for C in (10, 100):
        models["cluster_C%d" % C] = _capi.Engine(clusters=dict(n_clusters=C, cluster_type="mix", loss="Blackout"), **common)
    for e in models.values():       # small random parameters, identical stacks
        e.set_all_param_values([np.random.RandomState(1).normal(0, 0.05, s).astype(np.float32) for _, s in e.param_infos()])

    def step(name, e, i):
        X, mask, Y = data[i % len(data)]
        if name == "sampling":
            e.train_step_sampled(X, mask, Y, samples[i % 8], np.ones(B, np.float32))
        else:
            e.train_step_cluster(X, mask, Y, samples[i % 8], scale=1.0)

    times = {k: [] for k in models}
    for rnd in range(2):
        for name, e in (list(models.items()) if rnd == 0 else list(models.items())[::-1]):
            for i in range(args.warmup):
                step(name, e, i)
            e.timer_start()
            for i in range(args.steps):
                step(name, e, i)
            times[name].append(e.timer_stop() / args.steps)
    launches = {}
    for name, e in models.items():
        n0 = e.kernel_launches()
        step(name, e, 0)
        e.synchronize()
        launches[name] = e.kernel_launches() - n0
    res = {k: dict(ms_per_step=float(np.mean(v)), rounds_ms=[float(x) for x in v], kernel_launches_per_step=launches[k])
           for k, v in times.items()}
    base = res["sampling"]["ms_per_step"]
    for k in res:
        res[k]["overhead_vs_sampling"] = res[k]["ms_per_step"] / base - 1.0
    for e in models.values():
        e.close()
    return dict(shape="LSTM 2x256, N=50000, max_length=200, lengths U[100,200], B=512, S=32, Blackout, mix, Adam",
                steps=args.steps, warmup=args.warmup, results=res)


def topk(args):
    N, H, B, T, k = 500000, 512, 256, 20, 10
    rng = np.random.RandomState(2)
    data = batches(rng, 1, B, T, N, lo=5)[0]
    excl = [list(data[0][b, :int(data[1][b].sum()), 0]) for b in range(B)]
    out = {}
    for C, planted in ((10, True), (50, True), (200, True), (50, False)):
        e = _capi.Engine(n_items=N, cell="GRU", layers=(H,), max_length=T, batch_size=B, n_samples=1,
                         clusters=dict(n_clusters=C, cluster_type="mix", loss="Blackout"))
        vals = [np.random.RandomState(3).normal(0, 0.05, s).astype(np.float32) for _, s in e.param_infos()]
        if planted:
            R = -np.ones((N, C), np.float32)
            R[np.arange(N), rng.randint(0, C, N)] = 1.0
        else:
            R = (0.1 * rng.randn(N, C)).astype(np.float32)
        vals[-2] = R
        vals[-1] = rng.normal(0, 1.0, vals[-1].shape).astype(np.float32)
        e.set_all_param_values(vals)
        e.timer_start()
        sizes = e.cluster_build()
        build_ms = e.timer_stop()
        X, mask, _ = data

        def run(use):
            if use:
                return e.cluster_topk(X, mask, k=k, exclude=excl)
            return e.topk(X, mask, k=k, exclude=excl, neg_inf=True)

        ms = {}
        for use in (False, True, False, True):
            for _ in range(2):
                run(use)
            e.timer_start()
            for _ in range(args.steps):
                r = run(use)
            ms.setdefault("cluster" if use else "full", []).append(e.timer_stop() / args.steps)
        _, n, _ = e.cluster_topk(X, mask, k=k, exclude=excl)
        out["C%d_%s" % (C, "planted" if planted else "random")] = dict(
            full_topk_ms=float(np.mean(ms["full"])), cluster_topk_ms=float(np.mean(ms["cluster"])),
            speedup=float(np.mean(ms["full"]) / np.mean(ms["cluster"])), mean_items_scored=float(np.mean(n)),
            assr=float(N / np.mean(n)), cluster_build_ms=build_ms, largest_cluster=int(sizes.max()))
        e.close()
    return dict(shape="GRU 1x512 (H=512), N=500000, B=256 rows, max_length 20, k=10, ragged exclusion of the input items",
                note="R random (0.1 randn) puts every item in about half of the clusters: no reduction of the search "
                     "space; the planted partitions put each item in exactly one cluster",
                reps=args.steps, results=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", choices=["train", "topk"], default=None)
    args = ap.parse_args()
    if _capi.load_library().sbr_device_count() < 1:
        sys.exit("bench_cluster.py needs a CUDA device")
    res = dict(info=gpu_info())
    if args.only in (None, "train"):
        res["train_step"] = train_steps(args)
    if args.only in (None, "topk"):
        res["topk"] = topk(args)
    res["info_after"] = gpu_info()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        d = os.path.dirname(args.out)
        if d:
            os.makedirs(d, exist_ok=True)
        open(args.out, "w").write(txt)


if __name__ == "__main__":
    main()
