"""CPU: the RNNCluster oracle (tests/cluster_oracle.py) and host logic.

- float64 finite differences of the whole cluster step, every loss x cluster type, with separate cluster samples,
  selection noise and s != 1; the stack / out.* gradients equal those of the sampled loss without pop;
- an independent torch.autograd restatement of the reference expressions (rnn_cluster.py:151-251), h detached in the
  cluster branch;
- the scale schedule, prepare_tests against a literal transcription of rnn_cluster.py:464-480, the checkpoint file
  name, the nested save / load layout, the CLI dispatch and test.py's nb_of_dp handling.
"""
import argparse
import importlib.util
import os
import pickle

import numpy as np
import pytest

from oracle import sbr_oracle as O
from tests import cluster_oracle as CO
from tests.test_oracle import make_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, T, B, C = 23, 5, 4, 3


def _case(seed, cell="GRU", layers=(6,), sep=True, noise=True):
    rng = np.random.RandomState(seed)
    spec = O.Spec(n_items=N, cell=cell, layers=layers, loss="Blackout")
    vals = CO.init_params(spec, C, rng)
    for v in vals:
        if not v.any():
            v[...] = rng.normal(0, 0.1, size=v.shape)
    X, mask, _ = make_batch(rng, B, T, N, 1, 0)
    Y = rng.randint(0, N, size=B)
    samples = rng.randint(0, N, size=5)
    samples[0] = Y[1]
    cs = rng.randint(0, N, size=4) if sep else None
    nz = rng.normal(0, 0.3, size=(B, C)) if noise else None
    return spec, vals, X, mask, Y, samples, cs, nz


@pytest.mark.parametrize("ctype", CO.CLUSTER_TYPES)
@pytest.mark.parametrize("loss", CO.CLUSTER_LOSSES)
def test_oracle_finite_differences(loss, ctype):
    spec, vals, X, mask, Y, samples, cs, nz = _case(1, sep=(loss != "lin"), noise=(ctype != "sigmoid"))
    kw = dict(Y=Y, samples=samples, n_clusters=C, cluster_type=ctype, loss=loss, cluster_samples=cs, noise=nz, scale=1.6)
    c, cc, g = CO.cluster_loss_and_grads(spec, vals, X, mask, **kw)
    rng = np.random.RandomState(7)
    n_stack = len(vals) - 2
    for pi, v in enumerate(vals):
        for _ in range(3):
            idx = tuple(rng.randint(0, s) for s in v.shape)
            old = v[idx]
            eps = 1e-6
            v[idx] = old + eps
            cp, ccp, _ = CO.cluster_loss_and_grads(spec, vals, X, mask, **kw)
            v[idx] = old - eps
            cm, ccm, _ = CO.cluster_loss_and_grads(spec, vals, X, mask, **kw)
            v[idx] = old
            # stack and out.* see the recommendation cost only, Wc and R the cluster cost only
            num = (cp - cm) / (2 * eps) if pi < n_stack else (ccp - ccm) / (2 * eps)
            assert abs(num - g[pi][idx]) <= 1e-6 + 1e-5 * abs(num), (pi, idx, num, g[pi][idx])


@pytest.mark.parametrize("loss", ["Blackout", "BPR", "TOP1"])
def test_recommendation_branch_is_the_sampled_loss_without_pop(loss):
    spec, vals, X, mask, Y, samples, cs, nz = _case(2)
    _, _, g = CO.cluster_loss_and_grads(spec, vals, X, mask, Y=Y, samples=samples, n_clusters=C, loss=loss,
                                        cluster_samples=cs, noise=nz, scale=0.7)
    s2 = O.Spec(n_items=N, cell="GRU", layers=(6,), loss=loss)
    c0, g0 = O.loss_and_grads(s2, vals[:-2], X, mask, Y=Y, samples=samples, pop=np.ones(B))
    for a, b in zip(g[:-2], g0):
        np.testing.assert_allclose(a, b, rtol=1e-10, atol=1e-12)


def _torch_reference(loss, ctype, h, W, b, Wc, R, Y, samples, cs, noise, s):
    """rnn_cluster.py:151-251 written with torch ops, from the reference expressions."""
    import torch
    Bn = h.shape[0]
    t = torch.arange(Bn)

    def lossf(pred, n):
        if loss in ("Blackout", "CCE"):
            p = torch.softmax(pred, dim=-1)
            pos = -torch.log(p[t, t])
            return pos - torch.log(1 - p)[:, n:].sum(-1) if loss == "Blackout" else pos
        if loss == "lin":
            return pred[:, n:].sum(-1) - torch.diagonal(pred)
        diff = (pred - torch.diagonal(pred)[:, None])[:, n:]
        if loss == "BPR":
            return -torch.log(torch.sigmoid(-diff)).mean(-1)
        if loss == "BPRelu":
            x = diff + 0.5
            return (0.5 * 1.01 * x + 0.5 * 0.99 * torch.abs(x)).mean(-1)
        reg = pred[:, n:] ** 2
        return (torch.sigmoid(diff) + torch.sigmoid(reg)).mean(-1)

    cells = torch.cat([Y, samples])
    cost = lossf(h @ W[:, cells] + b[cells], Bn).mean()
    hd = h.detach()
    q = hd @ Wc + (noise if noise is not None else 0.0)
    sel = torch.softmax(q * s, dim=-1)
    rc = R[torch.cat([Y, cs])]
    if ctype == "softmax":
        m = torch.softmax(s * rc, dim=-1)
    elif ctype == "mix":
        m = torch.softmax(s * rc, dim=-1) + torch.sigmoid(s * rc)
    else:
        m = torch.sigmoid(s * rc)
    cost_c = lossf(sel @ m.T, Bn).mean()
    return cost, cost_c


@pytest.mark.parametrize("ctype", CO.CLUSTER_TYPES)
@pytest.mark.parametrize("loss", CO.CLUSTER_LOSSES)
def test_oracle_against_torch_autograd(loss, ctype):
    import torch
    spec, vals, X, mask, Y, samples, cs, nz = _case(3)
    c, cc, g = CO.cluster_loss_and_grads(spec, vals, X, mask, Y=Y, samples=samples, n_clusters=C, cluster_type=ctype,
                                         loss=loss, cluster_samples=cs, noise=nz, scale=1.3)
    P = O.as_dict(spec, vals[:-2])
    h, _ = O.forward_stack(spec, P, X, mask)
    ht = torch.tensor(h, requires_grad=True)
    W = torch.tensor(P["out.W"], requires_grad=True)
    b = torch.tensor(P["out.b"], requires_grad=True)
    Wc = torch.tensor(vals[-1], requires_grad=True)
    R = torch.tensor(vals[-2], requires_grad=True)
    cost, cost_c = _torch_reference(loss, ctype, ht, W, b, Wc, R, torch.tensor(Y), torch.tensor(samples),
                                    torch.tensor(cs), torch.tensor(nz), 1.3)
    (cost + cost_c).backward()
    assert abs(cost.item() - c) < 1e-10 and abs(cost_c.item() - cc) < 1e-10
    names = [n for n, _ in CO.param_names_shapes(spec, C)]
    np.testing.assert_allclose(g[names.index("out.W")], W.grad.numpy(), atol=1e-10)
    np.testing.assert_allclose(g[names.index("out.b")], b.grad.numpy(), atol=1e-10)
    np.testing.assert_allclose(g[-1], Wc.grad.numpy(), atol=1e-10)
    np.testing.assert_allclose(g[-2], R.grad.numpy(), atol=1e-10)
    # the gradient reaching h is the recommendation branch's alone
    _, dh_ref, _, _ = O.sampling_loss(O.Spec(n_items=N, loss="Blackout"), P, h, Y, samples, np.ones(B)) \
        if loss == "Blackout" else (None, None, None, None)
    if dh_ref is not None:
        np.testing.assert_allclose(ht.grad.numpy(), dh_ref, atol=1e-10)


def _transcribed_prepare_tests(cluster_membership):
    """rnn_cluster.py:464-480, line by line."""
    n_clusters = cluster_membership.shape[1]
    clusters = [[] for i in range(n_clusters)]
    for i in range(cluster_membership.shape[0]):
        no_cluster = True
        best_cluster = 0
        best_val = cluster_membership[i, 0]
        for j in range(n_clusters):
            if cluster_membership[i, j] > 0:
                clusters[j].append(i)
                no_cluster = False
            elif cluster_membership[i, j] > best_val:
                best_val = cluster_membership[i, j]
                best_cluster = j
        if no_cluster:
            clusters[best_cluster].append(i)
    return [np.array(c) for c in clusters]


def test_prepare_tests_matches_the_reference_loop():
    rng = np.random.RandomState(0)
    R = rng.randn(200, 7)
    R[:30] = -np.abs(R[:30])                # rows without a positive entry
    R[30:35] = -1.0                         # ties: the first arg-max
    for a, b in zip(CO.prepare_tests(R), _transcribed_prepare_tests(R)):
        np.testing.assert_array_equal(a, b)


def _cluster(**kw):
    from sbr_b200.neural_networks.rnn_cluster import RNNCluster
    from sbr_b200.neural_networks.recurrent_layers import RecurrentLayers
    from sbr_b200.neural_networks.update_manager import Adam
    return RNNCluster(recurrent_layer=RecurrentLayers(layer_type="GRU", layers=[50]), updater=Adam(), max_length=30,
                      batch_size=16, use_ratings_features=False, use_movies_features=False, use_users_features=False,
                      **kw)


def test_model_filename():
    p = _cluster(n_clusters=20, loss="CCE", sampling=32.0)
    common = p._common_filename(3)
    assert p._get_model_filename(3) == "rnn_clusters20_sc1.0_s32_mix_cCCE_" + common
    p = _cluster(n_clusters=5, loss="BPR", cluster_type="softmax", sampling=100, cluster_sampling=50, sampling_bias=0.5,
                 cluster_selection_noise=0.2, init_scale=2., scale_growing_rate=1.5, max_scale=20)
    assert p._get_model_filename(3) == "rnn_clusters5_sc2.0-1.5-20.0_p0.5s100_p0.5cs50_softmax_n0.2_cBPR_" + common
    p = _cluster(cluster_type="sigmoid", loss="lin")
    assert p._get_model_filename(1).startswith("rnn_clusters10_sc1.0_s100_cl")


def test_scale_schedule_follows_the_reference_rule():
    p = _cluster(init_scale=1.0, scale_growing_rate=2.0)

    class TS:
        epochs = 0.3
    p.dataset = argparse.Namespace(training_set=TS)

    def ref(state, epochs):   # rnn_cluster.py:398-405
        if 'last' not in state:
            state['last'] = epochs
        elif epochs > state['last'] + 1 and 2.0 != 1.:
            state['s'] *= 2.0 ** int(epochs - state['last'])
            state['last'] += int(epochs - state['last'])
        return state['s']
    st = dict(s=np.float32(1.0))
    for e in (0.3, 0.9, 1.2, 1.31, 1.5, 2.4, 4.9, 5.0, 8.2):
        TS.epochs = e
        p._update_scale()
        assert p.effective_scale == ref(st, e), e
    assert p.effective_scale > p.max_scale          # max_scale is stored, never applied
    q = _cluster(scale_growing_rate=1.0)
    q.dataset = p.dataset
    for e in (0.1, 3.0, 9.0):
        TS.epochs = e
        q._update_scale()
    assert q.effective_scale == 1.0


class _FakeEngine:
    def __init__(self, vals):
        self.vals = [np.asarray(v, np.float32) for v in vals]
        self.built = 0

    def get_all_param_values(self):
        return [v.copy() for v in self.vals]

    def set_all_param_values(self, vals):
        self.vals = [np.asarray(v, np.float32) for v in vals]

    def cluster_build(self):
        self.built += 1
        return np.zeros(3, np.int32)


def test_save_load_nested_layout(tmp_path):
    spec = O.Spec(n_items=N, layers=(6,))
    vals = CO.init_params(spec, C, np.random.RandomState(0))
    p = _cluster(n_clusters=C)
    p.engine = _FakeEngine(vals)
    f = str(tmp_path / "m" / "model.pkl")
    p.save(f)
    raw = pickle.load(open(f, "rb"))
    assert len(raw) == len(vals)
    np.testing.assert_array_equal(raw[-2], np.float32(vals[-2]))        # R
    assert isinstance(raw[-1], list) and len(raw[-1]) == 1               # [Wc]
    np.testing.assert_array_equal(raw[-1][0], np.float32(vals[-1]))
    q = _cluster(n_clusters=C)
    q.engine = _FakeEngine([np.zeros_like(v) for v in vals])
    q.load(f)
    for a, b in zip(q.engine.vals, vals):
        np.testing.assert_array_equal(a, np.float32(b))
    assert q.engine.built == 1                                           # load calls prepare_tests


def _args(argv):
    from sbr_b200.helpers import command_parser as parse
    return parse.command_parser(parse.predictor_command_parser, argv=argv)


@pytest.mark.parametrize("loss", ["CCE", "Blackout", "BPR", "TOP1", "BPRelu"])
def test_cli_builds_rnn_cluster(loss):
    from sbr_b200.helpers import command_parser as parse
    from sbr_b200.neural_networks.rnn_cluster import RNNCluster
    p = parse.get_predictor(_args(["--clusters", "5", "--loss", loss, "--ignore_clusters", "--c_sampling", "7"]))
    assert isinstance(p, RNNCluster) and p.loss == loss and p.n_clusters == 5 and not p.predict_with_clusters
    assert p.n_cluster_samples == 7 and p.n_samples == 32


def test_cli_cluster_errors_and_other_paths():
    from sbr_b200.helpers import command_parser as parse
    from sbr_b200.neural_networks.rnn_one_hot import RNNOneHot
    with pytest.raises(ValueError):
        parse.get_predictor(_args(["--clusters", "5", "--loss", "BPRI"]))
    with pytest.raises(ValueError):
        parse.get_predictor(_args(["--clusters", "5", "--loss", "hinge"]))
    with pytest.raises(ValueError):
        parse.get_predictor(_args(["--clusters", "5", "--sampling", "0.5"]))
    assert isinstance(parse.get_predictor(_args(["--loss", "CCE"])), RNNOneHot)


def _test_script():
    spec = importlib.util.spec_from_file_location("sbr_test_script", os.path.join(ROOT, "test.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


class _FakeDataset:
    n_items = 100

    def test_set(self, epochs=1):
        for u in range(4):
            yield np.array([[i, 5.0] for i in range(10 + u)]), u


class _FakePredictor:
    def __init__(self, clusters):
        self.clusters = clusters

    def load(self, f):
        pass

    def top_k_recommendations(self, seq, user_id=None, k=10):
        ids = list(range(20, 20 + k))
        return (ids, 10 + 10 * user_id) if self.clusters else ids


def test_test_py_sets_nb_of_dp_only_with_clusters(monkeypatch):
    ts = _test_script()
    monkeypatch.setattr(ts.evaluation, "Evaluator", lambda ds, k: argparse.Namespace(add_instance=lambda g, r: None))
    ev = ts.run_tests(_FakePredictor(True), "x", _FakeDataset(), argparse.Namespace(clusters=5), k=10)
    assert ev.nb_of_dp == np.mean([10, 20, 30, 40])
    ev = ts.run_tests(_FakePredictor(False), "x", _FakeDataset(), argparse.Namespace(clusters=-1), k=10)
    assert ev.nb_of_dp == 100
