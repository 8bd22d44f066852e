"""Golden fixture (tests/golden/c1_golden.npz, BASELINE.json config 1).

CPU: the oracle reproduces the frozen costs / final parameters / top-10 exactly (regression pin).
GPU: the CUDA path, through the C ABI, reproduces them within the parity tolerance: per-step cost
1e-4 absolute, parameters 2e-4, recall@10 and sps identical, top-10 lists >= 95% identical entries
(fp32 vs float64 near-ties may swap neighbours).

The fixture keeps the initial parameters as the seed of the oracle's initialisation plus the SHA-256 of
their bytes, and the final ones as int16-quantised steps from the initial ones (tests/golden/make_golden.py)."""
import hashlib
import os

import numpy as np
import pytest

from oracle import sbr_oracle as O

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c1_golden.npz"))
SPEC = O.Spec(n_items=500, cell="GRU", layers=(100,), loss="CCE")
NP = int(G["n_params"])


def _init():
    vals = O.init_params(SPEC, np.random.RandomState(int(G["init_seed"])), np.float32)
    digest = hashlib.sha256(b"".join(v.tobytes() for v in vals)).hexdigest()
    assert digest == str(G["init_sha256"]), "the seeded initialisation no longer gives the fixture's initial parameters"
    return vals


def _final(init):
    return [init[i].astype(np.float64) + G["final_q_%02d" % i] * float(G["final_scale_%02d" % i]) for i in range(NP)]


def _goals():
    off = G["val_goal_off"]
    return [list(G["val_goal_flat"][off[i]:off[i + 1]]) for i in range(len(off) - 1)]


def _seen():
    off = G["val_seen_off"]
    return [list(G["val_seen_flat"][off[i]:off[i + 1]]) for i in range(len(off) - 1)]


def test_oracle_reproduces_golden():
    init = _init()
    vals = [v.astype(np.float64) for v in init]
    upd = O.Updater("adam", lr=1e-3)
    for s in range(8):
        c = O.train_step(SPEC, vals, upd, G["X_%d" % s], G["mask_%d" % s], Y=G["Y_%d" % s], pop=G["pop_%d" % s].astype(np.float64))
        assert abs(float(c) - float(G["costs"][s])) < 1e-12
    for v, f in zip(vals, _final(init)):
        np.testing.assert_allclose(v, f, rtol=0, atol=1e-6)
    ex = np.zeros((len(G["val_X"]), 500))
    for i, s in enumerate(_seen()):
        ex[i, s] = 1
    top = O.top_k(O.test_scores(SPEC, vals, G["val_X"], G["val_mask"], exclude=ex), 10)
    np.testing.assert_array_equal(top, G["val_top10"])
    assert O.recall_at_k(_goals(), top, 10) == pytest.approx(float(G["val_recall10"]))


def test_float32_oracle_stays_within_parity_tolerance():
    """What a floatX=float32 Theano run would see: same fixture within 1e-4."""
    vals = _init()
    upd = O.Updater("adam", lr=1e-3)
    for s in range(8):
        c = O.train_step(SPEC, vals, upd, G["X_%d" % s], G["mask_%d" % s], Y=G["Y_%d" % s], pop=G["pop_%d" % s])
        assert abs(float(c) - float(G["costs"][s])) < 1e-4


@pytest.mark.gpu
def test_cuda_path_reproduces_golden():
    from sbr_b200 import _capi
    eng = _capi.Engine(n_items=500, cell="GRU", layers=(100,), loss="CCE", max_length=20, batch_size=20)
    try:
        init = _init()
        eng.set_all_param_values(init)
        for s in range(8):
            c = eng.train_step_cce(G["X_%d" % s], G["mask_%d" % s], G["Y_%d" % s], G["pop_%d" % s])
            assert abs(float(c) - float(G["costs"][s])) < 1e-4, (s, c, G["costs"][s])
        for v, f in zip(eng.get_all_param_values(), _final(init)):
            assert np.abs(v - f).max() < 2e-4
        top = eng.topk(G["val_X"], G["val_mask"], k=10, exclude=_seen())
        assert (top == G["val_top10"]).mean() >= 0.95
        goals = _goals()
        assert O.recall_at_k(goals, top, 10) == pytest.approx(float(G["val_recall10"]), abs=1e-4)
        assert float(np.mean([g[0] in t for g, t in zip(goals, top)])) == pytest.approx(float(G["val_sps"]), abs=1e-4)
    finally:
        eng.close()
