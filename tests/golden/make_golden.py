"""Generate tests/golden/c1_golden.npz -- the frozen parity fixture for BASELINE.json config 1
(RNNOneHot GRU-1x100, 500 items, 200 users, seq-len<=20, batch 16).

The reference (Python 2 + Theano + Lasagne) cannot be run in this environment, so the fixture is
produced by the float64 numpy oracle (oracle/sbr_oracle.py), whose gradients are pinned by
finite differences and by torch.autograd (tests/test_oracle*.py).  PARITY UNPINNED against the real
reference; regenerate with   python tests/golden/make_golden.py   (deterministic, ~2 s).

Contents: the initial parameters (float32, checkpoint order) as the seed of oracle.init_params and the
SHA-256 of their bytes, 8 training batches built by the host mirror of RNNBase._gen_mini_batch on a
seeded synthetic dataset, the per-step costs of 8 Adam steps (float64), the parameters after those
steps, and for 20 validation users the input, the goal and the oracle's top-10 + recall@10 / sps after
training.  Stored whole, the random initial and final parameters would not fit in 1 MB; so each final
parameter is kept as its step from the initial one, quantised to int16 over the largest step
(final = init + final_q * final_scale, within final_scale / 2 ~ 1.2e-7 of the float64 oracle).
"""
import hashlib
import os
import random
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import sbr_oracle as O  # noqa: E402


def init_sha256(vals):
    return hashlib.sha256(b"".join(np.ascontiguousarray(v, np.float32).tobytes() for v in vals)).hexdigest()


def build():
    from sbr_b200.helpers import synthetic
    from sbr_b200.helpers.data_handling import DataHandler
    from sbr_b200.neural_networks.recurrent_layers import RecurrentLayers
    from sbr_b200.neural_networks.rnn_one_hot import RNNOneHot
    from sbr_b200.neural_networks.update_manager import Adam
    d = tempfile.mkdtemp(prefix="sbr_golden_")
    path = synthetic.write_dataset(os.path.join(d, "c1"), 200, 500, seed=1234, uniform_len=(5, 40))
    ds = DataHandler(path)
    pred = RNNOneHot(recurrent_layer=RecurrentLayers(layer_type="GRU", layers=[100]), updater=Adam(), max_length=20,
                     batch_size=16, use_ratings_features=False, use_movies_features=False, use_users_features=False)
    pred.n_items = ds.n_items
    pred.set_dataset(ds)
    random.seed(1234)
    np.random.seed(1234)
    gen = pred._gen_mini_batch(ds.training_set())
    batches = [next(gen) for _ in range(8)]
    spec = O.Spec(n_items=500, cell="GRU", layers=(100,), loss="CCE")
    init_seed = 1
    init32 = O.init_params(spec, np.random.RandomState(init_seed), np.float32)
    vals = [v.astype(np.float64) for v in init32]
    upd = O.Updater("adam", lr=1e-3)
    costs = []
    for X, mask, Y, pop, _ in batches:
        costs.append(float(O.train_step(spec, vals, upd, X, mask, Y=Y, pop=pop.astype(np.float64))))
    # validation instances (test=True split in the middle)
    vgen = pred._gen_mini_batch(ds.validation_set(epochs=1), test=True)
    VX, VM, goals, seen = [], [], [], []
    for (X, mask, Y, pop, excl), goal in vgen:
        VX.append(X[0]); VM.append(mask[0]); goals.append(goal); seen.append(excl[0])
    VX, VM = np.stack(VX), np.stack(VM)
    ex = np.zeros((len(VX), 500))
    for i, s in enumerate(seen):
        ex[i, s] = 1
    top = O.top_k(O.test_scores(spec, vals, VX, VM, exclude=ex), 10)
    recall = O.recall_at_k(goals, top, 10)
    sps = float(np.mean([g[0] in t for g, t in zip(goals, top)]))
    out = {"n_params": len(init32), "costs": np.array(costs), "val_X": VX, "val_mask": VM, "val_top10": top,
           "val_recall10": recall, "val_sps": sps,
           "val_goal_flat": np.concatenate([np.asarray(g, np.int32) for g in goals]),
           "val_goal_off": np.cumsum([0] + [len(g) for g in goals]).astype(np.int32),
           "val_seen_flat": np.concatenate([np.asarray(s, np.int32) for s in seen]),
           "val_seen_off": np.cumsum([0] + [len(s) for s in seen]).astype(np.int32)}
    out["init_seed"] = init_seed
    out["init_sha256"] = init_sha256(init32)
    for i, (a, b) in enumerate(zip(init32, vals)):
        step = b - a.astype(np.float64)
        scale = np.abs(step).max() / 32767 or 1.0
        out["final_q_%02d" % i] = np.round(step / scale).astype(np.int16)
        out["final_scale_%02d" % i] = scale
    for i, (X, mask, Y, pop, _) in enumerate(batches):
        out["X_%d" % i] = X; out["mask_%d" % i] = mask; out["Y_%d" % i] = Y; out["pop_%d" % i] = pop
    return out


if __name__ == "__main__":
    out = build()
    dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c1_golden.npz")
    np.savez_compressed(dst, **out)
    print("wrote", dst, os.path.getsize(dst), "bytes; costs", out["costs"], "recall@10", out["val_recall10"])
