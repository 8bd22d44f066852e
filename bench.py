#!/usr/bin/env python
"""bench.py -- training throughput of the RNN hot path in user-sequences/sec.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config c1|c2|c3|c4|c5]
                    [--dump-outputs DIR]

A "step" is one call of the reference's `train_function(*batch)` (neural_networks/rnn_base.py:290):
gather -> recurrent scan -> output projection + loss -> BPTT -> scatter -> (all-reduce) -> Adam, on one
synthetic mini-batch.  Default workload (BASELINE.json configs[1], the configuration `metric` is quoted
on): RNNOneHot, LSTM 1x200, MovieLens-1M-shaped synthetic data (6040 users, 3706 items, mean
sequence length ~165), max_length 200, 128 rows per GPU, Adam, fp32.  `--config c3|c4|c5` select the other
BASELINE.json shapes with the reference's own losses (C3 RNNSampling BPR S=32; C4 RNNMargin hinge over the full
catalog; C5 RNNOneHot GRU 2x512 over 500k items), per-GPU rows = the global batch BASELINE names / its GPU count.
Batches come from the host mirror of `_gen_mini_batch` (nested prefixes of one user's sequence).

One JSON line on stdout (rank 0):
  value      whole-job sequences/sec with the batches already resident in HBM (device slots),
             timed on the device with a cudaEvent pair on the library's stream, max over ranks;
  e2e        the same metric through the public API (`RNNOneHot.train_function(X, mask, Y, pop)`)
             with HOST numpy buffers: pinned staging + H2D of the inputs and the D2H read of the
             cost are inside the timed region of every step;
  roofline   the dominant kernel (largest stage of the step), algorithmic FLOPs / its measured
             launch time, against MEASURED_PEAKS.json;
  cpu_baseline  the numpy restatement of the reference's Theano CPU path (oracle/, "port") timed on
             this box's host cores on a bounded sample of the same batches (rank 0, N=1 only);
  valid_steps_per_s  valid (row, step) pairs per second over all ranks: the global batches of N ranks hold longer
             rows, this number separates that workload shift from overhead in a scaling curve;
  per_rank   (N > 1) every rank's scan time and the valid steps of its slice -- a straggler is visible;
  multi_rank_cost_check  (N > 1, C1/C2) the all-reduced global cost of step 0 against a one-rank replay of the same
             global batch; parity / parity_max_abs (N = 1) the step-0 cost against the CPU port.

The device-timed region holds exactly K = --steps steps.  Without --steps, K is the config's `steps`, chosen for about
1 s of device time on one B200 (C2: 2000 steps, 1.30 s on a B200 at its 1000 W power limit and 1965 MHz), so the
window is long enough to average out the clock and the scheduler and for the clock sampler to see the load.  The K
steps cycle over min(K, MAX_BATCHES) distinct batches (timed step i uses batch W + i % that), so a large K needs no
more host-built batches or HBM slots.  Before the timed region run W warm-up steps and one untimed pass over those
batches, so the number of steps before the last timed one depends only on the arguments.

`--dump-outputs DIR` (e.g. bench_outputs/<build>, which git ignores) then writes what the last timed step computed --
its cost and the parameters it left, as a caller of train_function sees them -- to DIR/*.npy (see dump_outputs).  The
inputs are seeded, so the dumps of two builds compare output for output.  The library sums gradients with
floating-point atomics, and Adam turns the rounding differences of near-zero gradients into full-size steps, so
trajectories drift apart with the step count: two runs of one build on C2 agree to 1e-5 after W=5 and K=20, but not
after the default K=2000 (median parameter difference 0.05).  Compare builds on a short run such as --steps 20.

`--impl reference` times that CPU restatement alone (the reference itself -- Python 2 + Theano +
Lasagne -- cannot be installed here; see DESIGN.md) with all host threads numpy's BLAS will use.  It runs every one
of its K steps (default REFERENCE_STEPS) with no time limit; on an 8-core Xeon host a step took 1.7 s for C2 (128
rows), 6.9 s for C4 and 12.2 s for C5 (16 rows each, gradients only), plus the synthetic data set on first use.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: model + data shape; B = rows per GPU (weak scaling), gpus = the GPU count BASELINE.json quotes it on;
    # steps = the default --steps of the B200 arm, about 1 s of device time on one B200 (ms/step in profiles/README.md;
    # C1 0.125 ms/step measured)
    "c1": dict(label="C1 RNNOneHot GRU-1x100, 500 items, 200 users, seq-len<=20, batch 16",
               model="onehot", loss="CCE", cell="GRU", layers=(100,), n_items=500, n_users=200, T=20, B=16,
               uniform_len=(5, 40), gpus=1, steps=8000),
    "c2": dict(label="C2 RNNOneHot LSTM-1x200, ML-1M shape (3706 items, 6040 users, mean len 165), max_length 200, "
                     "batch 128/GPU, full softmax + CCE, Adam",
               model="onehot", loss="CCE", cell="LSTM", layers=(200,), n_items=3706, n_users=6040, T=200, B=128,
               uniform_len=None, gpus=1, steps=2000),
    "c3": dict(label="C3 RNNSampling BPR (S=32; 'BPR-max' does not exist in the reference) LSTM-2x256, 50k items, "
                     "max_length 200, batch 512/GPU, Adam",
               model="sampling", loss="BPR", S=32, cell="LSTM", layers=(256, 256), n_items=50000, n_users=6040, T=200,
               B=512, uniform_len=None, gpus=1, steps=120),
    "c4": dict(label="C4 RNNMargin hinge over the full catalog (the reference has no sampled-target margin) "
                     "LSTM-1x512, 200k items, max_length 200, batch 1024 over 4 GPUs = 256/GPU, Adam",
               model="margin", loss="hinge", cell="LSTM", layers=(512,), n_items=200000, n_users=6040, T=200, B=256,
               uniform_len=None, gpus=4, steps=120),
    "c5": dict(label="C5 RNNOneHot GRU-2x512, 500k items, max_length 500, batch 2048 over 8 GPUs = 256/GPU, full "
                     "softmax + CCE, Adam",
               model="onehot", loss="CCE", cell="GRU", layers=(512, 512), n_items=500000, n_users=6040, T=500, B=256,
               uniform_len=None, gpus=8, steps=60),
}
MAX_BATCHES = 128     # distinct batches the timed steps cycle over: timed step i uses batch W + i % min(K, MAX_BATCHES)
REFERENCE_STEPS = 5   # default --steps of the reference arm (seconds per step on the host, see the docstring)


def timed_batches(W, K):
    """Batch indices of the K timed steps."""
    nb = min(K, MAX_BATCHES)
    return [W + i % nb for i in range(K)]


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------------------------
# workload
# ----------------------------------------------------------------------------------------------
def make_dataset(cfg):
    from sbr_b200.helpers import synthetic
    from sbr_b200.helpers.data_handling import DataHandler
    tag = "sbr_bench_%d_%d_%s" % (cfg["n_users"], cfg["n_items"], "u" if cfg["uniform_len"] else "ln")
    d = os.path.join(tempfile.gettempdir(), tag)
    if not os.path.exists(os.path.join(d, "data", "stats")):
        tmp = d + ".%d.tmp" % os.getpid()
        kw = dict(uniform_len=cfg["uniform_len"]) if cfg["uniform_len"] else {}
        synthetic.write_dataset(tmp, cfg["n_users"], cfg["n_items"], seed=1234, **kw)
        try:
            os.rename(tmp, d)
        except OSError:
            pass  # another rank won the race
    return DataHandler(d + "/")


def make_predictor(cfg, dataset, n_ranks=1, rank=0, nccl_id=None, device=0, n_slots=1, create_engine=True,
                   rows_per_gpu=None):
    from sbr_b200.neural_networks.recurrent_layers import RecurrentLayers
    from sbr_b200.neural_networks.update_manager import Adam
    B = rows_per_gpu or cfg["B"]
    common = dict(recurrent_layer=RecurrentLayers(layer_type=cfg["cell"], layers=list(cfg["layers"])),
                  updater=Adam(), max_length=cfg["T"], batch_size=B * n_ranks,
                  use_ratings_features=False, use_movies_features=False, use_users_features=False,
                  device=device, n_ranks=n_ranks, rank=rank, nccl_id=nccl_id, init_seed=1)
    if cfg["model"] == "onehot":
        from sbr_b200.neural_networks.rnn_one_hot import RNNOneHot
        p = RNNOneHot(**common)
    elif cfg["model"] == "sampling":
        from sbr_b200.neural_networks.rnn_sampling import RNNSampling
        p = RNNSampling(loss_function=cfg["loss"], sampling=cfg["S"], **common)
    else:
        from sbr_b200.neural_networks.rnn_margin import RNNMargin
        p = RNNMargin(loss_function=cfg["loss"], **common)
    base = p._engine_extra_kwargs
    p._engine_extra_kwargs = lambda: dict(base(), n_slots=n_slots)
    if create_engine:
        p.prepare_model(dataset)
    else:
        p.n_items = dataset.n_items
        if cfg["model"] == "sampling":
            p.effective_sampling = int(cfg["S"])
    p.set_dataset(dataset)
    return p


def make_batches(predictor, dataset, n):
    """n global mini-batches from the host mirror of _gen_mini_batch (same on every rank)."""
    random.seed(1234)
    np.random.seed(1234)
    devnull = open(os.devnull, "w")
    stdout, sys.stdout = sys.stdout, devnull      # "Opening file (n)" chatter of the generator
    try:
        gen = predictor._gen_mini_batch(dataset.training_set())
        return [next(gen) for _ in range(n)]
    finally:
        sys.stdout = stdout
        devnull.close()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, cost, names, params):
    """cost.npy (float64 [1]) and one float32 param_<ii>_<name>.npy per parameter, at most DUMP_LIMIT_BYTES in all.
    When the parameters do not fit, each one larger than an equal share of the limit is replaced by a sample of its
    flattened entries at indices drawn from RandomState(<ii>) (file name ending in .sample), the same in every run."""
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "cost.npy"), np.array([cost], np.float64))
    room = (DUMP_LIMIT_BYTES - 4096 * (len(params) + 1)) // 4      # float32 entries; 4 KB per file for its header
    share = room // len(params)
    sample = sum(p.size for p in params) > room
    for i, (name, p) in enumerate(zip(names, params)):
        fname = "param_%02d_%s" % (i, name)
        a = np.asarray(p, np.float32)
        if sample and a.size > share:
            idx = np.sort(np.random.RandomState(i).randint(0, a.size, share))
            a, fname = a.reshape(-1)[idx], fname + ".sample"
        np.save(os.path.join(dirname, fname + ".npy"), a)


def n_out_columns(cfg, B_global):
    return cfg["n_items"] if cfg["model"] != "sampling" else B_global + cfg["S"]


def step_work(cfg, batch, n_ranks):
    """Algorithmic work of one step on this global batch (SURVEY.md §8d), per GPU: forward FLOPs =
    sum_layers 2*V*H*G*H (+ 2*V*I*G*H input GEMM for layers >= 1) + 2*B*H*C, step = 3 x forward; V = valid (b, t)
    pairs.  Per-stage figures feed the per-kernel rooflines."""
    mask = batch[1]
    V = float(mask.sum()) / n_ranks
    B = mask.shape[0] / n_ranks
    G = 4 if cfg["cell"] == "LSTM" else (3 if cfg["cell"] == "GRU" else 1)
    rec = inp = 0.0
    prev = None
    for H in cfg["layers"]:
        rec += 2.0 * V * H * G * H
        if prev is not None:
            inp += 2.0 * V * prev * G * H
        prev = H
    C = n_out_columns(cfg, mask.shape[0])
    out = 2.0 * B * cfg["layers"][-1] * C
    H0 = cfg["layers"][0]
    return {"step_flops": 3.0 * (rec + inp + out), "V": V,
            "flops": {"rnn_fwd": rec + inp, "rnn_bwd": rec + inp, "wgrad": rec + inp, "output": 3.0 * out},
            "bytes": {"gather": 2.0 * V * G * H0 * 4, "scatter": V * G * H0 * 4}}


# ----------------------------------------------------------------------------------------------
# CPU arm: numpy restatement of the reference graph (oracle/), float32 like a tuned Theano run
# ----------------------------------------------------------------------------------------------
def oracle_spec(cfg):
    from oracle import sbr_oracle as O
    return O.Spec(n_items=cfg["n_items"], cell=cfg["cell"], layers=tuple(cfg["layers"]), loss=cfg["loss"])


def oracle_kwargs(cfg, pred, batch, rows=None):
    """The oracle's view of a batch made by the host mirror's _prepare_input (first `rows` rows)."""
    sl = slice(0, rows)
    if cfg["model"] == "onehot":
        X, mask, Y, pop, _ = batch
        return X[sl], mask[sl], dict(Y=Y[sl], pop=pop[sl])
    if cfg["model"] == "sampling":
        X, mask, Y, samples, pop, _ = batch
        return X[sl], mask[sl], dict(Y=Y[sl], samples=samples, pop=pop[sl])
    X, mask, (off, ids), w, seen = batch
    n = len(w) if rows is None else min(rows, len(w))
    Ym, Wm = pred.dense_targets((X[:n], mask[:n], (off[:n + 1], ids), w[:n], seen[:n]))
    return X[:n], mask[:n], dict(Ymat=Ym, Wmat=Wm)


def cpu_reference_rate(cfg, pred, batches, steps, warmup, rows=None, budget_s=25.0, vals=None, update=True):
    """sequences/s of the numpy restatement on `rows` rows per step (None = the whole batch)."""
    from oracle import sbr_oracle as O
    spec = oracle_spec(cfg)
    if vals is None:
        vals = O.init_params(spec, np.random.RandomState(1), np.float32)
    upd = O.Updater("adam", lr=1e-3)
    times, costs = [], []
    t_begin = time.perf_counter()
    for i in range(warmup + steps):
        X, mask, kw = oracle_kwargs(cfg, pred, batches[i % len(batches)], rows)
        t0 = time.perf_counter()
        if update:
            cost = O.train_step(spec, vals, upd, X, mask, **kw)
        else:
            cost, _ = O.loss_and_grads(spec, vals, X, mask, **kw)
        dt = time.perf_counter() - t0
        if not np.isfinite(cost):
            raise RuntimeError("oracle cost is not finite")
        costs.append(float(cost))
        if i >= warmup:
            times.append(dt)
        if time.perf_counter() - t_begin > budget_s and len(times) >= 1:
            break
    n_rows = X.shape[0]
    mean = float(np.mean(times))
    return n_rows / mean, mean, len(times), n_rows, costs


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        n = [p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"]
        return max(n) if n else 1
    except Exception:
        return os.cpu_count() or 1


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default: the config's 'steps' for the B200 arm, %d for the reference arm)"
                         % REFERENCE_STEPS)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--rows-per-gpu", type=int, default=0, help="override the per-GPU batch of the config")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the cost and the parameters left by the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the B200 path computed; it needs --impl b200")
    cfg = dict(CONFIGS[args.config])
    if args.rows_per_gpu > 0:
        cfg["B"] = args.rows_per_gpu
    W = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    K = args.steps if args.steps is not None else (cfg["steps"] if args.impl == "b200" else REFERENCE_STEPS)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        log("warning: WORLD_SIZE=%d but --gpus %d; using WORLD_SIZE" % (world, args.gpus))
    n_gpus = world if world > 1 else 1
    if args.impl == "reference":
        n_gpus = max(world, args.gpus)      # describes the same global batch as the B200 arm at this N
    B_global = cfg["B"] * n_gpus
    staged = cfg["model"] == "onehot"       # device-resident batch slots exist for the CCE step (sbr_stage_cce)

    base = {"metric": "user-sequences/sec (training step, device-timed)", "unit": "sequences/s", "n_gpus": n_gpus,
            "steps": K, "warmup": W, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic (ML-1M-shaped, seed 1234), random-init weights",
            "config": {"workload": cfg["label"], "global_batch": B_global, "seq_len": cfg["T"],
                       "parallelism": "dp%d" % n_gpus,
                       "l2": "no explicit flush: a step streams more activation bytes than the 126 MB L2 and every "
                             "timed step uses a different batch"}}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        dataset = make_dataset(cfg)
        pred = make_predictor(cfg, dataset, n_ranks=n_gpus, create_engine=False)
        batches = make_batches(pred, dataset, min(K + W, 8))
        # a step = the first `rows` rows of the global mini-batch (bounded sample of the same workload)
        rows = min(B_global, 128 if args.config in ("c1", "c2") else (64 if args.config == "c3" else 16))
        heavy = args.config in ("c4", "c5")      # 0.5-1 G parameters: gradients only, no Adam pass over the arena
        rate, sec, done, n_rows, _ = cpu_reference_rate(cfg, pred, batches, K, W, rows=rows, budget_s=float("inf"),
                                                        update=not heavy)
        cores = blas_threads()
        out = dict(base)
        out.update({"impl": "reference", "value": rate, "ms_per_step": sec * 1e3, "steps": done, "gpu_launches": 0,
                    "cpu_baseline": {"value": rate, "unit": "sequences/s", "cores": cores, "kind": "port",
                                     "sample": "%d steps of %d rows (of the %d-row global batch) of the numpy float32 "
                                               "restatement of the reference's Theano CPU graph%s, BLAS threads=%d of "
                                               "%d host cores; Theano/Lasagne (Python 2) cannot be installed here"
                                               % (done, n_rows, B_global, " (gradients only)" if heavy else "", cores,
                                                  os.cpu_count())},
                    "e2e": {"value": rate, "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        print(json.dumps(out))
        return 0

    # ------------------------------------------------------------------ B200 arm
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
        os.environ["NCCL_DEBUG"] = "NONE"       # stdout carries exactly one JSON line (NCCL prints its banner there)
    from sbr_b200 import _capi
    from sbr_b200.helpers.rendezvous import Control
    ctl = Control() if n_gpus > 1 else None        # TCP control plane; the gradients use the library's NCCL
    nccl_id = ctl.broadcast(_capi.nccl_unique_id() if rank == 0 else None) if ctl else None

    dataset = make_dataset(cfg)
    timed = timed_batches(W, K)
    n_batches = W + min(K, MAX_BATCHES)
    pred = make_predictor(cfg, dataset, n_ranks=n_gpus, rank=rank, nccl_id=nccl_id, device=local_rank,
                          n_slots=n_batches if staged else 1)
    pred._compile_train_function()
    eng = pred.engine
    batches = make_batches(pred, dataset, n_batches)
    vals0 = eng.get_all_param_values() if (rank == 0 and args.config in ("c1", "c2", "c3")) else None

    def barrier():
        if ctl:
            ctl.barrier()

    def max_over_ranks(x):
        return ctl.all_max(x) if ctl else x

    def run_steps(idx, want_cost=False):
        c = None
        for i in idx:
            if staged:
                c = eng.train_step_staged(i, want_cost=want_cost)
            else:
                c = pred.train_function(*batches[i])
        return c

    # ---- leg 1: device-timed; CCE batches resident in HBM (device slots) ------------------------------
    if staged:
        for i, b in enumerate(batches):
            X, mask, Y, pop, _ = b
            sl = pred._split_rows
            eng.stage_cce(i, sl(X), sl(mask), sl(Y), sl(pop))
    step0_cost = None
    if staged:
        step0_cost = float(eng.train_step_staged(0, want_cost=True))     # global cost of the first step (parity checks)
        run_steps(range(1, W))
    else:
        step0_cost = float(pred.train_function(*batches[0]))
        run_steps(range(1, W))
    eng.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.15)      # nvidia-smi needs ~0.1 s before its first sample
    barrier()
    # one untimed pass over the batches of the timed region warms every batch shape it uses; it runs after the
    # sampler's start-up sleep, so the device is not left idle between the warm pass and the timed steps
    t_enq = time.perf_counter()
    run_steps(range(W, n_batches))
    host_enqueue_ms = (time.perf_counter() - t_enq) * 1e3 / (n_batches - W)     # host enqueue time of a step
    launches0 = eng.kernel_launches()
    eng.timer_start()
    run_steps(timed)
    ms = eng.timer_stop()
    barrier()
    launches = eng.kernel_launches() - launches0
    last_cost = eng.synchronize(want_cost=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, float(last_cost), [n for n, _ in eng.param_infos()], eng.get_all_param_values())
    ms = max_over_ranks(ms)
    value = B_global * K / (ms * 1e-3)

    # ---- leg 2: end to end through the public API, host buffers ------------------------------
    for i in range(min(W, 3)):
        pred.train_function(*batches[i])
    eng.synchronize()
    barrier()
    t0 = time.perf_counter()
    for i in timed:
        cost = pred.train_function(*batches[i])
    eng.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    clocks = sampler.stop() if rank == 0 else None     # sampled across both timed legs
    barrier()
    e2e_value = B_global * K / e2e_s
    Bl, T = cfg["B"], cfg["T"]
    h2d = Bl * T * 4 + Bl * 4 * 3
    if cfg["model"] == "sampling":
        h2d += (B_global + cfg["S"]) * 4
    d2h = 4

    # ---- leg 3: per-stage device times (separate pass; profiling syncs every step) -------------
    eng.set_profiling(True)
    acc = {}
    for i in timed:
        if staged:
            eng.train_step_staged(i, want_cost=False)
        else:
            pred.train_function(*batches[i])
        for k, v in eng.stage_times().items():
            acc[k] = acc.get(k, 0.0) + v / K
    eng.set_profiling(False)
    works = [step_work(cfg, batches[i], n_gpus) for i in timed]
    mean_V = float(np.mean([w["V"] for w in works]))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_bw = peaks.get("hbm_gbs", 6500.0)
    peak_src = "MEASURED_PEAKS.json (bf16_tflops_sustained, hbm_gbs; measured)" if peaks else "fallback 1.4 PFLOP/s / 6.5 TB/s"
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    P = eng.total_params()
    stage_alg = {}      # stage -> (bound, algorithmic flops or bytes per step)
    for k in ("rnn_fwd", "rnn_bwd", "wgrad", "output"):
        stage_alg[k] = ("tensor", float(np.mean([w["flops"][k] for w in works])))
    for k in ("gather", "scatter"):
        stage_alg[k] = ("hbm", float(np.mean([w["bytes"][k] for w in works])))
    stage_alg["optimizer"] = ("hbm", 32.0 * P)
    kernels = {"rnn_fwd": "rnn_fwd_tc_kernel / tc_gemm_kernel<*_FWD> (+ input GEMMs)", "rnn_bwd": "rnn_bwd_tc_kernel / tc_gemm_kernel<*_BWD>",
               "wgrad": "wgrad_tc_kernel / tc_gemm_kernel<STORE> (weight + input gradients)", "output": "tc_gemm_kernel<STORE> x3 + loss kernel",
               "gather": "gather_rows_kernel", "scatter": "scatter_add_rows_kernel", "optimizer": "optimizer_kernel"}

    def roof(stage):
        bound, alg = stage_alg[stage]
        t_ms = acc.get(stage, 0.0)
        if t_ms <= 0:
            return None
        if bound == "tensor":
            a = alg / (t_ms * 1e-3) / 1e12
            return {"kernel": kernels[stage], "stage": stage, "bound": "tensor", "achieved": a, "peak": peak_tf,
                    "unit": "TFLOP/s", "frac": a / peak_tf, "frac_of_3xtf32_peak": a / (peak_tf / 6.0),
                    "traffic": traffic.get(stage), "algorithmic_flops_per_step": alg, "stage_ms": t_ms}
        a = alg / (t_ms * 1e-3) / 1e9
        return {"kernel": kernels[stage], "stage": stage, "bound": "hbm", "achieved": a, "peak": peak_bw, "unit": "GB/s",
                "frac": a / peak_bw, "traffic": traffic.get(stage), "algorithmic_bytes_per_step": alg, "stage_ms": t_ms}

    ranked = sorted((k for k in stage_alg if acc.get(k, 0.0) > 0), key=lambda k: -acc[k])
    roofs = [r for r in (roof(k) for k in ranked[:3]) if r]
    roofline = dict(roofs[0]) if roofs else None
    if roofline:
        roofline.update({"peak_source": peak_src,
                         "math": "3xTF32 on tcgen05 (fp32-accurate): 3 MMA passes at the TF32 rate = 1/6 of the bf16 "
                                 "peak per algorithmic FLOP",
                         "valid_steps_per_launch": mean_V, "stage_ms_all": {k: round(v, 4) for k, v in acc.items()}})

    # every rank's own scan time and valid (row, step) pairs of its slice (rows r = rank mod N): the straggler is visible
    per_rank = None
    if ctl:
        try:
            my_valid = float(np.mean([np.asarray(batches[i][1])[rank::n_gpus].sum() for i in timed]))
        except Exception:
            my_valid = None
        per_rank = ctl.all_gather({"rank": rank, "scan_ms": round(acc.get("rnn_fwd", 0.0) + acc.get("rnn_bwd", 0.0), 4),
                                   "all_stages_ms": round(sum(acc.values()), 4), "valid_steps": my_valid})

    out = None
    if rank == 0:
        out = dict(base)
        if per_rank is not None:
            out["per_rank"] = sorted(per_rank, key=lambda e: e["rank"])
        out.update({"impl": "b200", "value": value, "ms_per_step": ms / K,
                    "host_enqueue_ms_per_step": host_enqueue_ms, "clocks": clocks,
                    "valid_steps_per_s": mean_V * n_gpus * K / (ms * 1e-3),
                    "value_inputs": "device-resident batch slots" if staged else
                                    "host buffers through train_function (no device slots for this loss): H2D inside",
                    "e2e": {"value": e2e_value, "unit": "sequences/s", "h2d_bytes_per_step": h2d * n_gpus,
                            "d2h_bytes_per_step": d2h * n_gpus, "ms_per_step": e2e_s / K * 1e3},
                    "gpu_launches": int(launches) * n_gpus, "roofline": roofline, "roofline_top3": roofs,
                    "last_cost": float(last_cost), "e2e_last_cost": float(cost), "step0_cost": step0_cost})
        if vals0 is not None and not args.no_cpu_baseline:
            # CPU leg: the numpy restatement from the SAME initial parameters on the SAME first batch -> parity of the
            # step-0 cost, then a few timed steps
            full = n_gpus == 1 and args.config in ("c1", "c2")
            rows = None if full else min(B_global, 64)
            from oracle import sbr_oracle as O
            spec = oracle_spec(cfg)
            if n_gpus == 1:
                X, mask, kw = oracle_kwargs(cfg, pred, batches[0], None)
                c_ref, _ = O.loss_and_grads(spec, [v.astype(np.float32) for v in vals0], X, mask, **kw)
                out["parity_max_abs"] = abs(float(c_ref) - step0_cost)
                out["parity"] = {"step0_cost_b200": step0_cost, "step0_cost_cpu_port": float(c_ref),
                                 "tolerance": 1e-4, "ok": bool(abs(float(c_ref) - step0_cost) <= 1e-4)}
                rate, sec, done, n_rows, _ = cpu_reference_rate(cfg, pred, batches[:4], 6, 1, rows=rows, budget_s=25.0)
                cores = blas_threads()
                out["cpu_baseline"] = {"value": rate, "unit": "sequences/s", "cores": cores, "kind": "port",
                                       "sample": "%d steps of %d rows (batch %d) of the numpy float32 restatement of the "
                                                 "reference graph, %.2f s/step, BLAS threads=%d of %d host cores; "
                                                 "Python-loop bound (as fast with 1 BLAS thread)"
                                                 % (done, n_rows, B_global, sec, cores, os.cpu_count())}
    if n_gpus > 1 and staged and args.config in ("c1", "c2"):
        # multi-rank correctness inside the run: rank 0 replays step 0 of the same GLOBAL batch on a single-rank engine
        # from the same initial parameters; the all-reduced global cost must match
        if rank == 0:
            p1 = make_predictor(cfg, dataset, n_ranks=1, device=local_rank, rows_per_gpu=B_global)
            p1.engine.set_all_param_values(vals0)
            X, mask, Y, pop, _ = batches[0]
            c1 = float(p1.engine.train_step_cce(X, mask, Y, pop))
            p1.engine.close()
            out["multi_rank_cost_check"] = {"global_cost_n_ranks": step0_cost, "single_rank_replay": c1,
                                            "abs_diff": abs(c1 - step0_cost), "ok": bool(abs(c1 - step0_cost) <= 1e-4)}
        barrier()
    if rank == 0:
        print(json.dumps(out))
    eng.close()
    if ctl:
        ctl.barrier()
        ctl.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
