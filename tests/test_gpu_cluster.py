"""GPU: RNNCluster (sbr_create_cluster and friends) against the float64 cluster oracle (tests/cluster_oracle.py).
Tolerances as in test_gpu_parity: cost and cluster cost within 1e-4, every gradient within 2e-4 * max|g| + 1e-7,
parameters within 2e-4 after a few optimizer steps."""
import argparse
import os
import random

import numpy as np
import pytest

from oracle import sbr_oracle as O
from tests import cluster_oracle as CO
from tests.test_oracle import make_batch

pytestmark = pytest.mark.gpu

N, T, B = 150, 9, 13     # B is not a multiple of the 8 / 16-row scan tiles


def _engine(spec, C, ctype, loss, n_cs=0, **kw):
    from sbr_b200 import _capi
    args = dict(n_items=spec.n_items, cell=spec.cell, layers=spec.layers, max_length=T, batch_size=B,
                bidirectional=spec.bidirectional, n_samples=7,
                clusters=dict(n_clusters=C, cluster_type=ctype, loss=loss, n_cluster_samples=n_cs))
    args.update(kw)
    return _capi.Engine(**args)


def _setup(spec, C, seed, sep_cs, noise):
    rng = np.random.RandomState(seed)
    vals = CO.init_params(spec, C, rng)
    for v in vals:
        if not v.any():
            v[...] = rng.normal(0, 0.05, size=v.shape)
    X, mask, _ = make_batch(rng, B, T, N, 1, 0)
    Y = rng.randint(0, N, size=B)
    samples = rng.randint(0, N, size=7)
    samples[:3] = Y[:3]                        # samples that collide with targets
    cs = rng.randint(0, N, size=5) if sep_cs else None
    if cs is not None:
        cs[0] = Y[4]
    nz = rng.normal(0, 0.3, size=(B, C)) if noise else None
    return vals, X, mask, Y, samples, cs, nz


def _close_grads(g, r):
    for a, b in zip(g, r):
        tol = 2e-4 * np.abs(b).max() + 1e-7
        assert np.abs(a - b).max() <= tol, (np.abs(a - b).max(), tol)


# (cell, layers, bidirectional, C, loss, type, separate cluster samples, noise, scale)
CASES = [
    ("GRU", (24,), False, 7, "Blackout", "mix", True, True, 1.7),
    ("LSTM", (24,), False, 2, "CCE", "mix", False, False, 1.0),
    ("Vanilla", (24,), False, 64, "BPR", "mix", True, True, 0.6),
    ("GRU", (16, 24), False, 7, "TOP1", "mix", False, True, 2.0),
    ("LSTM", (16,), True, 7, "BPRelu", "mix", True, False, 1.3),
    ("GRU", (24,), False, 64, "lin", "mix", False, False, 1.0),
    ("LSTM", (24,), False, 7, "Blackout", "softmax", True, True, 1.5),
    ("GRU", (24,), False, 2, "Blackout", "sigmoid", False, True, 0.8),
]


@pytest.mark.parametrize("cell,layers,bi,C,loss,ctype,sep,noise,scale", CASES)
def test_cluster_step_matches_oracle(cell, layers, bi, C, loss, ctype, sep, noise, scale):
    spec = O.Spec(n_items=N, cell=cell, layers=layers, bidirectional=bi, loss="Blackout")
    vals, X, mask, Y, samples, cs, nz = _setup(spec, C, 3, sep, noise)
    c0, cc0, g0 = CO.cluster_loss_and_grads(spec, vals, X, mask, Y=Y, samples=samples, n_clusters=C, cluster_type=ctype,
                                            loss=loss, cluster_samples=cs, noise=nz, scale=scale)
    eng = _engine(spec, C, ctype, loss, n_cs=5 if sep else 0)
    try:
        names = [n for n, _ in eng.param_infos()]
        assert names == [n for n, _ in CO.param_names_shapes(spec, C)]
        eng.set_all_param_values(vals)
        eng.set_skip_update(True)
        cost, ccost = eng.train_step_cluster(X, mask, Y, samples, cluster_samples=cs, noise=nz, scale=scale)
        assert abs(float(cost) - c0) < 1e-4
        assert abs(float(ccost) - cc0) < 1e-4
        _close_grads(eng.get_all_grads(), g0)
    finally:
        eng.close()


@pytest.mark.parametrize("kind,steps", [("adam", 5), ("adagrad", 3)])
def test_cluster_trajectory_matches_two_updaters(kind, steps):
    """One fused update over the arena == the reference's two updater instances (rnn_cluster.py:265-270)."""
    spec = O.Spec(n_items=N, cell="GRU", layers=(24,), loss="Blackout")
    C = 7
    vals, X, mask, Y, samples, cs, nz = _setup(spec, C, 5, True, True)
    lr = 1e-2
    eng = _engine(spec, C, "mix", "Blackout", n_cs=5, updater=kind, lr=lr)
    try:
        eng.set_all_param_values(vals)
        u_rec, u_clu = O.Updater(kind, lr=lr), O.Updater(kind, lr=lr)
        rng = np.random.RandomState(9)
        for s in range(steps):
            samples = rng.randint(0, N, size=7)
            cs = rng.randint(0, N, size=5)
            cost, ccost = eng.train_step_cluster(X, mask, Y, samples, cluster_samples=cs, noise=nz, scale=1.3)
            c0, cc0, g = CO.cluster_loss_and_grads(spec, vals, X, mask, Y=Y, samples=samples, n_clusters=C,
                                                   cluster_type="mix", loss="Blackout", cluster_samples=cs, noise=nz,
                                                   scale=1.3)
            u_rec.step(vals[:-2], g[:-2])
            u_clu.step(vals[-2:][::-1], g[-2:][::-1])     # [Wc, R], the reference's order
            assert abs(float(cost) - c0) < 1e-4 and abs(float(ccost) - cc0) < 1e-4, s
        for a, b in zip(eng.get_all_param_values(), vals):
            assert np.abs(a - b).max() < 2e-4
    finally:
        eng.close()


def _planted(spec, C, seed):
    """Parameters whose R gives clusters of very different sizes, one smaller than k, and items with no positive
    entry (they fall back to their row's arg-max)."""
    rng = np.random.RandomState(seed)
    vals = CO.init_params(spec, C, rng)
    R = -np.abs(rng.normal(0.5, 0.2, size=(N, C)))
    owner = rng.randint(1, C, size=N)
    owner[:3] = 0                               # cluster 0: 3 items (< k)
    R[np.arange(N), owner] = np.abs(rng.normal(0.5, 0.2, size=N))
    R[10:20, :] = -np.abs(rng.normal(0.5, 0.2, size=(10, C)))     # no positive entry
    R[25:40, (owner[25:40] + 1) % C] = 0.3       # some items in two clusters
    R[3:, 0] = -5.0                              # ... and no other item in cluster 0, not even as a fallback
    vals[-2] = R
    # let every cluster be selected by some row
    vals[-1] = rng.normal(0, 1.0, size=vals[-1].shape)
    return rng, vals


def _check_ids(ids, scores, k):
    """GPU ids against oracle scores: the picked ids carry the k best scores (robust to ties)."""
    best = np.sort(scores)[::-1][:k]
    got = scores[ids]
    both_inf = np.isneginf(best) & np.isneginf(got)
    assert np.all(both_inf | (np.abs(got - best) <= 1e-4 * np.abs(best).max() + 1e-6)), (got, best)
    assert len(set(ids.tolist())) == len(ids)


@pytest.mark.parametrize("ctype", ["mix", "softmax", "sigmoid"])
def test_cluster_test_topk_and_restricted_topk(ctype):
    spec = O.Spec(n_items=N, cell="LSTM", layers=(32,), loss="Blackout")
    C, k = 6, 10
    rng, vals = _planted(spec, C, 11)
    X, mask, lens = make_batch(rng, B, T, N, 1, 0)
    excl = [list(X[b, :lens[b], 0]) for b in range(B)]
    exd = np.zeros((B, N))
    for b in range(B):
        exd[b, excl[b]] = 1
    eng = _engine(spec, C, ctype, "Blackout")
    try:
        eng.set_all_param_values(vals)
        full, clus, sel, used = eng.cluster_test_topk(X, mask, k=k, exclude=excl)
        s1, s2, c, n_used = CO.cluster_test_scores(spec, vals, X, mask, C, ctype, exclude=exd)
        np.testing.assert_array_equal(sel, c)
        np.testing.assert_allclose(used, n_used, rtol=1e-4, atol=1e-3)
        for b in range(B):
            _check_ids(full[b], s1[b], k)
            _check_ids(clus[b], s2[b], k)
        # prepare_tests on the device
        sizes = eng.cluster_build()
        ref = CO.prepare_tests(vals[-2])
        np.testing.assert_array_equal(sizes, [len(x) for x in ref])
        assert sizes[0] == 3
        # cluster-restricted top-k; excluded ids and clusters smaller than k
        ids, n, sel2 = eng.cluster_topk(X, mask, k=k, exclude=excl, use_clusters=True)
        np.testing.assert_array_equal(sel2, c)
        for b, (items, sc, nd) in enumerate(CO.cluster_topk_scores(spec, vals, X, mask, ref, exclude=excl)):
            assert n[b] == nd
            keff = min(k, nd)
            assert np.all(ids[b, keff:] == -1)
            pos = np.searchsorted(items, ids[b, :keff])
            assert np.all(items[pos] == ids[b, :keff])
            _check_ids(pos, sc, keff)
        # every member of a small cluster is returned when k covers it
        small = np.nonzero(sizes <= k)[0]
        rows = [b for b in range(B) if sel2[b] in small]
        ids_nx, n_nx, _ = eng.cluster_topk(X, mask, k=k, exclude=None)
        for b in rows:
            assert sorted(ids_nx[b, :n_nx[b]].tolist()) == ref[sel2[b]].tolist()
        # --ignore_clusters: the whole catalog
        ids_f, n_f, _ = eng.cluster_topk(X, mask, k=k, exclude=excl, use_clusters=False)
        assert np.all(n_f == N)
        for b, (items, sc, _) in enumerate(CO.cluster_topk_scores(spec, vals, X, mask, ref, exclude=excl,
                                                                  use_clusters=False)):
            _check_ids(ids_f[b], sc, k)
    finally:
        eng.close()


@pytest.fixture(scope="module")
def dataset(tmp_path_factory):
    from sbr_b200.helpers import synthetic
    from sbr_b200.helpers.data_handling import DataHandler
    d = tmp_path_factory.mktemp("ds")
    return DataHandler(synthetic.write_dataset(str(d / "c1"), 200, 500, seed=1234, uniform_len=(5, 40)))


def test_rnn_cluster_trains_reports_metrics_and_tests(dataset, tmp_path):
    """The CLI builds RNNCluster; a short training run returns finite costs and every cluster metric; the saved model
    round-trips through load and test.py's run_tests reports assr = N / mean cluster size."""
    import importlib.util
    spec_ = importlib.util.spec_from_file_location("sbr_test_script", os.path.join(os.path.dirname(os.path.dirname(
        os.path.abspath(__file__))), "test.py"))
    test_script = importlib.util.module_from_spec(spec_)
    spec_.loader.exec_module(test_script)
    from sbr_b200.helpers import command_parser as parse
    from sbr_b200.neural_networks.rnn_cluster import RNNCluster
    args = parse.command_parser(parse.predictor_command_parser, argv=[
        "--clusters", "5", "--loss", "Blackout", "--r_t", "GRU", "--r_l", "32", "-b", "16", "--max_length", "20",
        "--sampling", "16", "--c_sampling", "12", "--csn", "0.1", "--scale_growing_rate", "1.5", "--u_m", "adam"])
    p = parse.get_predictor(args)
    assert isinstance(p, RNNCluster)
    p.prepare_model(dataset)
    random.seed(3); np.random.seed(3)
    costs = []
    p._compile_train_function()
    orig = p.train_function
    p.train_function = lambda *b: costs.append(orig(*b)) or costs[-1]
    metrics, _, best = p.train(dataset, max_iter=60, progress=30, autosave='All', save_dir=str(tmp_path) + "/",
                               validation_metrics=['sps'])
    assert len(costs) == 60 and np.all(np.isfinite(costs))
    assert np.isfinite(p.last_cluster_cost)
    for m in p.metrics:
        assert metrics[m] is not None, m
    assert metrics['assr'] >= 1.0 and len(metrics['cluster_use']) == 5
    # save / load in the nested layout, then test.py's evaluation loop
    import pickle
    saved = pickle.load(open(best, "rb"), encoding="latin1")
    assert len(saved) == len(p.engine.param_infos()) and isinstance(saved[-1], list) and len(saved[-1]) == 1
    q = parse.get_predictor(args)
    q.prepare_model(dataset)
    q.set_dataset(dataset)
    q.load(best)
    flat = saved[:-2] + [saved[-2], saved[-1][0]]
    for a, b in zip(q.engine.get_all_param_values(), flat):
        np.testing.assert_array_equal(a, b)
    ev = test_script.run_tests(q, best, dataset, argparse.Namespace(clusters=5), k=10)
    ns = [q.top_k_recommendations(s[:len(s) // 2], k=10)[1] for s, _ in dataset.test_set(epochs=1)]
    assert ev.assr() == pytest.approx(dataset.n_items / np.mean(ns))
    assert all(n in set(q.cluster_sizes.tolist()) for n in ns)
    p.engine.close(); q.engine.close()


_RANK_SCRIPT = r"""
import sys, pickle
sys.path.insert(0, sys.argv[1])
import torch.distributed as dist
from sbr_b200 import _capi
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
box = [_capi.nccl_unique_id() if rank == 0 else None]
dist.broadcast_object_list(box, src=0)
d = pickle.load(open(sys.argv[2], "rb"))
Bl = d["B"] // world
eng = _capi.Engine(n_items=d["N"], cell="LSTM", layers=(32,), max_length=d["T"], batch_size=Bl, device=rank, n_ranks=world,
                   rank=rank, nccl_id=box[0], global_batch=d["B"], n_samples=8,
                   clusters=dict(n_clusters=5, cluster_type="mix", loss="Blackout", n_cluster_samples=6))
eng.set_all_param_values(d["vals"])
lo = rank * Bl
out = []
for X, mask, Y, samples, cs, nz in d["batches"]:
    out.append(tuple(float(c) for c in eng.train_step_cluster(X[lo:lo+Bl], mask[lo:lo+Bl], Y[lo:lo+Bl], samples, cs,
                                                                nz[lo:lo+Bl], 1.4, Y_all=Y, row_offset=lo)))
pickle.dump((out, eng.get_all_param_values()), open(sys.argv[2] + ".out%d" % rank, "wb"))
eng.close()
dist.barrier()
dist.destroy_process_group()
"""


def test_two_rank_cluster_matches_single_rank(tmp_path):
    """2 ranks, global batch split by rows (noise sliced by rows too): both costs are global, replicas stay equal and
    follow the single-process oracle."""
    import pickle
    import subprocess
    import sys
    from sbr_b200 import _capi
    if _capi.load_library().sbr_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    rng = np.random.RandomState(4)
    Nn, Tt, Bb, C = 300, 12, 16, 5
    spec = O.Spec(n_items=Nn, cell="LSTM", layers=(32,), loss="Blackout")
    vals = [v.astype(np.float32) for v in CO.init_params(spec, C, rng)]
    batches = []
    for _ in range(3):
        X, mask, _ = make_batch(rng, Bb, Tt, Nn, 1, 0)
        batches.append((X, mask, rng.randint(0, Nn, Bb).astype(np.int32), rng.randint(0, Nn, 8).astype(np.int32),
                        rng.randint(0, Nn, 6).astype(np.int32), rng.normal(0, 0.2, (Bb, C)).astype(np.float32)))
    f = str(tmp_path / "job.pkl")
    pickle.dump(dict(N=Nn, T=Tt, B=Bb, vals=vals, batches=batches), open(f, "wb"))
    script = str(tmp_path / "rank.py")
    open(script, "w").write(_RANK_SCRIPT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29733", script, root, f]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    r0 = pickle.load(open(f + ".out0", "rb")); r1 = pickle.load(open(f + ".out1", "rb"))
    for a, b in zip(r0[1], r1[1]):
        np.testing.assert_array_equal(a, b)
    assert r0[0] == r1[0]
    v64 = [v.astype(np.float64) for v in vals]
    u_rec, u_clu = O.Updater("adam", lr=1e-3), O.Updater("adam", lr=1e-3)
    for s, (X, mask, Y, samples, cs, nz) in enumerate(batches):
        c0, cc0, g = CO.cluster_loss_and_grads(spec, v64, X, mask, Y=Y, samples=samples, n_clusters=C, cluster_type="mix",
                                               loss="Blackout", cluster_samples=cs, noise=nz.astype(np.float64), scale=1.4)
        u_rec.step(v64[:-2], g[:-2])
        u_clu.step(v64[-2:], g[-2:])
        assert abs(r0[0][s][0] - c0) < 1e-4 and abs(r0[0][s][1] - cc0) < 1e-4
    for a, b in zip(v64, r0[1]):
        assert np.abs(a - b).max() < 2e-4
