"""GPU parity sweep over every recurrent-scan kernel variant the dispatcher can pick.

Each case is written for specific variants: the test first asserts that the live plan of every layer and direction
(sbr_plan_layer_scan on the engine's handle) is exactly that variant, so a retuned heuristic fails here instead of
silently moving the case elsewhere, and that one step launches exactly the planned number of scan kernels
(sbr_scan_launches).  It then compares, against the float64 oracle,
  - the forward alone: scores, rtol 2e-4;
  - the cost (1e-4) and every gradient tensor (2e-4 * max|g| + 1e-7), as test_gpu_parity.check_grads does;
  - every hidden-unit ownership slice the plans report (tcgen05 / FFMA CTA slices [r*Hs, min(H, (r+1)*Hs)), the 8-unit
    forward and 128-unit backward tiles of the persistent scans) of every parameter with a hidden-unit axis, against
    its own scale: err <= 2e-4 * max|g_slice| + 2e-5 * max|g_tensor| + 1e-7.  A slice of small gradients (the last CTA
    of H = 200 owns 4 units) is then not hidden behind the largest value of the whole tensor.

Every batch has a row of length T, a row of length 1 and random lengths in between; T = 9 wraps the 4-stage TMA rings
of the tcgen05 scans.  Cases with B % 16 == 0 on tcgen05 layers also run wgrad_tc_kernel.

CASES is plain data: tests/test_scan_dispatch.py checks on the CPU that the cases reach every variant the planner
can return on a B200.
"""
import zlib

import numpy as np
import pytest

from oracle import sbr_oracle as O

N_ITEMS = 97
T_DEFAULT = 9
G_OF = {"LSTM": 4, "GRU": 3, "Vanilla": 1}


def variant(plan, backward):
    """Canonical name of the kernel variant in a plan (a dict from _capi.plan_layer_scan)."""
    d = "bwd" if backward else "fwd"
    f, G = plan["family"], plan["G"]
    if f == "tc_cluster":
        return ("tc", d, G, plan["MT"], plan["BT"]) if backward else ("tc", d, G, plan["BT"])
    if f == "ffma":
        return ("ffma", d, G, plan["BT"], plan["JU"], bool(plan["wsmem"]))
    if f == "persistent":
        return ("persistent", d, G, ("splitk" if plan["splitk"] else "nosplit") if backward else "launch")
    return ("step", d, G)


def _case(cid, cell, layers, B, expect, env=None, T=T_DEFAULT, sliced=False):
    """expect: per layer (forward variant, backward variant).  sliced: the top layer's persistent scans need at least
    two launches in each direction (batch tiles beyond what one co-resident launch holds)."""
    return dict(id=cid, cell=cell, layers=tuple(layers), B=B, T=T, env=dict(env or {}), sliced=sliced,
                expect=[tuple(e) for e in expect])


def _tc(G, H, bt):
    return (("tc", "fwd", G, bt), ("tc", "bwd", G, 1 if H <= 128 else 2, bt))


def _ff(G, fwd, bwd):
    return (("ffma", "fwd", G) + fwd, ("ffma", "bwd", G) + bwd)


def _pers(G, bwd="splitk"):
    return (("persistent", "fwd", G, "launch"), ("persistent", "bwd", G, bwd))


def _step(G):
    return (("step", "fwd", G), ("step", "bwd", G))


CASES = []
# tcgen05 cluster scans: both tile heights; H = 8 is the smallest shape they take (C = 2, Hs = 4), 128 the largest with
# one 128-unit backward tile, 144 the first with two (its last CTA owns 4 of 20 units), 224 fills both TMEM budgets
for _cell in ("LSTM", "GRU", "Vanilla"):
    for _H in (8, 128, 144, 224):
        for _bt in (8, 16):
            CASES.append(_case("tc-%s%d-bt%d" % (_cell, _H, _bt), _cell, (_H,), 32, [_tc(G_OF[_cell], _H, _bt)],
                               env={"SBR_TC_BT": str(_bt)}))
    for _H in (144, 224):      # partial 16-row tile; the weight gradient comes from tc_gemm instead of wgrad_tc
        CASES.append(_case("tc-%s%d-B13" % (_cell, _H), _cell, (_H,), 13, [_tc(G_OF[_cell], _H, 16)]))
# the rectifier (a Vanilla layer fed by a dense input) on the tcgen05 scans
CASES.append(_case("tc-relu224", "Vanilla", (48, 224), 32, [_tc(1, 48, 8), _tc(1, 224, 8)], env={"SBR_TC_BT": "8"}))
CASES.append(_case("tc-relu8", "Vanilla", (48, 8), 32, [_tc(1, 48, 16), _tc(1, 8, 16)], env={"SBR_TC_BT": "16"}))

# FFMA cluster scans, one case per reachable <G, BT, JU, WSMEM> at natural shapes: H % 4 != 0, or H % 16 != 0 above
# 224, or one of the holes of tc_plan (140, 196).  16-row tiles from B > 144, 32-row tiles from B > 288 (8 CTAs).
_BT16 = {"SBR_TC_BT": "16"}     # pins the tile height of the tcgen05 layer 0 of the Vanilla stacks
CASES += [
    _case("ffma-LSTM50", "LSTM", (50,), 13, [_ff(4, (8, 1, True), (8, 1, True))]),
    _case("ffma-LSTM196-B200", "LSTM", (196,), 200, [_ff(4, (16, 1, True), (16, 1, True))]),
    _case("ffma-LSTM140-B300", "LSTM", (140,), 300, [_ff(4, (32, 1, True), (32, 1, True))]),
    _case("ffma-LSTM264", "LSTM", (264,), 13, [_ff(4, (8, 2, True), (8, 2, True))]),
    # the 16-row JU = 2 forward tile does not fit next to the LSTM weight slice: the forward stays at 8 rows
    _case("ffma-LSTM264-B200", "LSTM", (264,), 200, [_ff(4, (8, 2, True), (16, 2, True))]),
    _case("ffma-LSTM500", "LSTM", (500,), 13, [_ff(4, (8, 2, False), (8, 2, False))]),
    _case("ffma-LSTM500-B200", "LSTM", (500,), 200, [_ff(4, (16, 2, False), (16, 2, False))]),
    _case("ffma-GRU37", "GRU", (37,), 13, [_ff(3, (8, 1, True), (8, 1, True))]),
    _case("ffma-GRU140-B200", "GRU", (140,), 200, [_ff(3, (16, 1, True), (16, 1, True))]),
    _case("ffma-GRU140-B320", "GRU", (140,), 320, [_ff(3, (32, 1, True), (32, 1, True))]),
    _case("ffma-GRU264", "GRU", (264,), 13, [_ff(3, (8, 2, True), (8, 2, True))]),
    _case("ffma-GRU264-B200", "GRU", (264,), 200, [_ff(3, (16, 2, True), (16, 2, True))]),
    _case("ffma-GRU500", "GRU", (500,), 13, [_ff(3, (8, 2, False), (8, 2, False))]),
    _case("ffma-GRU500-B200", "GRU", (500,), 200, [_ff(3, (16, 2, False), (16, 2, False))]),
    _case("ffma-relu50", "Vanilla", (48, 50), 13, [_tc(1, 48, 16), _ff(1, (8, 1, True), (8, 1, True))]),
    _case("ffma-relu140-B200", "Vanilla", (48, 140), 200, [_tc(1, 48, 16), _ff(1, (16, 1, True), (16, 1, True))], env=_BT16),
    _case("ffma-relu140-B320", "Vanilla", (48, 140), 320, [_tc(1, 48, 16), _ff(1, (32, 1, True), (32, 1, True))], env=_BT16),
    _case("ffma-relu264", "Vanilla", (48, 264), 13, [_tc(1, 48, 16), _ff(1, (8, 2, True), (8, 2, True))]),
    _case("ffma-relu264-B200", "Vanilla", (48, 264), 200, [_tc(1, 48, 16), _ff(1, (16, 2, True), (16, 2, True))], env=_BT16),
]

# persistent scans: one 128-row forward tile per 148 / (H / 8) SMs and 32-row split-K backward tiles per co-resident
# cluster slot, so these batches need a second launch (tile0 > 0) in both directions
_NOSPLIT = {"SBR_DISABLE_SPLITK_SCAN": "1"}
CASES += [
    _case("pers-GRU512-B300", "GRU", (512,), 300, [_pers(3)], sliced=True),
    _case("pers-LSTM320-B400", "LSTM", (320,), 400, [_pers(4)], sliced=True),
    _case("pers-relu320-B400", "Vanilla", (48, 320), 400, [_tc(1, 48, 16), _pers(1)], env=_BT16, sliced=True),
    _case("pers-GRU512-B1200-nosplit", "GRU", (512,), 1200, [_pers(3, "nosplit")], env=_NOSPLIT, sliced=True),
    _case("pers-LSTM320-nosplit", "LSTM", (320,), 40, [_pers(4, "nosplit")], env=_NOSPLIT),
    _case("pers-relu320-nosplit", "Vanilla", (48, 320), 40, [_tc(1, 48, 16), _pers(1, "nosplit")], env=dict(_NOSPLIT, **_BT16)),
]

# per-step tensor-core scans (what H % 16 == 0 above 224 runs without the persistent kernels)
_NOPERS = {"SBR_DISABLE_PERSISTENT_SCAN": "1"}
CASES += [
    _case("step-LSTM256", "LSTM", (256,), 40, [_step(4)], env=_NOPERS),
    _case("step-GRU256", "GRU", (256,), 40, [_step(3)], env=_NOPERS),
    _case("step-relu256", "Vanilla", (48, 256), 40, [_tc(1, 48, 16), _step(1)], env=dict(_NOPERS, **_BT16)),
]


def scan_batch(rng, B, T, N):
    """Rows of length T and 1 first, then random lengths."""
    lens = rng.randint(1, T + 1, size=B)
    lens[0], lens[1] = T, 1
    X = np.zeros((B, T, 1), dtype=np.int32)
    mask = np.zeros((B, T))
    for b in range(B):
        X[b, :lens[b], 0] = rng.randint(0, N, size=lens[b])
        mask[b, :lens[b]] = 1
    return X, mask, lens


def slices(plan):
    return [(r * plan["Hs"], (r + 1) * plan["Hs"]) for r in range(plan["C"])]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c["id"] for c in CASES])
def test_scan_variant_against_oracle(case, monkeypatch):
    from tests.test_gpu_parity import _engine, _init
    for k, v in case["env"].items():
        monkeypatch.setenv(k, v)
    spec = O.Spec(n_items=N_ITEMS, cell=case["cell"], layers=case["layers"], loss="CCE")
    B, T = case["B"], case["T"]
    rng, vals = _init(spec, zlib.crc32(case["id"].encode()))
    X, mask, lens = scan_batch(rng, B, T, N_ITEMS)
    Y, pop = rng.randint(0, N_ITEMS, size=B), rng.uniform(0.5, 2.0, size=B)
    eng = _engine(spec, B, T)
    try:
        eng.set_all_param_values(vals)
        eng.set_skip_update(True)
        # 1. the live plans are the variants this case was written for
        plans = [(eng.plan_layer_scan(case["cell"], H, B, False, lens, T), eng.plan_layer_scan(case["cell"], H, B, True, lens, T))
                 for H in case["layers"]]
        got = [(variant(f, False), variant(b, True)) for f, b in plans]
        assert got == case["expect"], "plan moved: %s" % got
        if case["sliced"]:
            f, b = plans[-1]
            assert f["launches"] >= 2 and b["launches"] >= 2, (f, b)
        n_fwd = sum(f["launches"] for f, _ in plans)
        n_bwd = sum(b["launches"] for _, b in plans)
        # 2. the forward alone, and its scan launches
        n0 = eng.scan_launches()
        s = eng.scores(X, mask)
        assert eng.scan_launches() - n0 == n_fwd
        np.testing.assert_allclose(s, O.scores(spec, vals, X, mask), rtol=2e-4, atol=1e-7)
        # 3. one training step: cost and gradients
        n0 = eng.scan_launches()
        cost = eng.train_step_cce(X, mask, Y, pop)
        grads = eng.get_all_grads()
        assert eng.scan_launches() - n0 == n_fwd + n_bwd
        c0, g0 = O.loss_and_grads(spec, vals, X, mask, Y=Y, pop=pop)
        assert abs(float(cost) - float(c0)) <= 1e-4, (cost, c0)
        names = [n for n, _ in O.param_names_shapes(spec)]
        for name, a, g in zip(names, g0, grads):
            tol = 2e-4 * np.abs(a).max() + 1e-7
            err = np.abs(a - g).max()
            assert err <= tol, "%s: max err %.3e > tol %.3e" % (name, err, tol)
        # 4. every ownership slice against its own scale
        for li, (H, (pf, pb)) in enumerate(zip(case["layers"], plans)):
            for name, a, g in zip(names, g0, grads):
                if not name.startswith("l%d." % li):
                    continue
                assert a.shape[-1] == H, name
                scale = np.abs(a).max()
                for lo, hi in sorted(set(slices(pf) + slices(pb))):
                    if lo >= H:
                        continue
                    sa, sg = a[..., lo:hi], g[..., lo:hi]
                    tol = 2e-4 * np.abs(sa).max() + 2e-5 * scale + 1e-7
                    err = np.abs(sa - sg).max()
                    assert err <= tol, "%s units [%d, %d): max err %.3e > tol %.3e (slice scale %.3e, tensor %.3e)" % (
                        name, lo, min(hi, H), err, tol, np.abs(sa).max(), scale)
    finally:
        eng.close()
