"""CPU: the recurrent-scan dispatch table (sbr_plan_layer_scan, the planner the scan launchers decide with).

- the family every hidden size 1..512 runs on a B200, pinned literally (any change of the dispatch rule shows in a diff);
- the set of kernel variants the planner can return equals the set of template cases the dispatch code compiles
  (rnn_tc.cu SBR_FWD_CASE / SBR_BWD_CASE, rnn_cluster.cu SBR_FFMA_FWD / SBR_FFMA_BWD, the persistent launches of
  tc_scan.cu, the step epilogues of tc_gemm.cu): no variant is compiled that nothing can run, none is reachable
  without a kernel;
- the cases of tests/test_gpu_scan_variants.py plan to the variants they are written for and cover every one.
B200 description: 148 SMs, 15 co-resident 8-CTA tcgen05 clusters, 37 co-resident 4-CTA split-K clusters.
"""
import os
import re

import pytest

from tests.test_gpu_scan_variants import CASES, scan_batch, variant

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "sequence-based-recommendations_b200", "csrc")
SWITCHES = ("SBR_DISABLE_TC", "SBR_DISABLE_TC_BWD", "SBR_DISABLE_STEP_SCAN", "SBR_DISABLE_PERSISTENT_SCAN",
            "SBR_DISABLE_SPLITK_SCAN", "SBR_DISABLE_TC_GEMM", "SBR_DISABLE_TMA_GEMM", "SBR_SCAN_MULTICAST", "SBR_TC_BT",
            "SBR_TC_FORCE_MIXED", "SBR_TC_NO_MIXED")

# family of every H = 1..512 (row k holds H = 64k+1 .. 64k+64), the same for the three cells and both directions:
# T tcgen05 cluster scans, P persistent scans, F FFMA cluster scans
FAMILY_PIN = (
    "FFFFFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFT"
    "FFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFT"
    "FFFFFFFFFFFFFFFTFFFTFFFTFFFTFFFTFFFFFFFFFFFTFFFTFFFTFFFTFFFTFFFT"
    "FFFFFFFTFFFTFFFTFFFTFFFTFFFTFFFTFFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFP"
    "FFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFP"
    "FFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFP"
    "FFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFP"
    "FFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFPFFFFFFFFFFFFFFFP"
)
# H % 4 == 0 and 8 <= H <= 224, but tc_plan finds no cluster split (C = 8: Hs * 7 >= H; C = 4: Hs > 32)
TC_HOLES = [132, 136, 140, 164, 168, 196]
LETTER = {"tc_cluster": "T", "persistent": "P", "ffma": "F", "step": "S"}


@pytest.fixture
def clean_env(monkeypatch):
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    return monkeypatch


def plan(cell, H, B, backward, lens=None, t_max=10):
    from sbr_b200 import _capi
    return _capi.plan_layer_scan(cell, H, B, backward, lens=lens, t_max=t_max)


def test_family_of_every_hidden_size_is_pinned(clean_env):
    for cell in ("LSTM", "GRU", "Vanilla"):
        for backward in (False, True):
            got = "".join(LETTER[plan(cell, H, 32, backward)["family"]] for H in range(1, 513))
            assert got == FAMILY_PIN, (cell, backward)
    assert [H for H in range(8, 225, 4) if FAMILY_PIN[H - 1] != "T"] == TC_HOLES


def test_cluster_split_at_the_edges(clean_env):
    """(C, Hs) of the tcgen05 scans at the smallest accepted H, the largest single-tile backward, the first two-tile
    backward (last CTA owns 4 units) and the largest accepted H (forward 64 + 2*224 = 512 TMEM columns, backward
    32*2 + 2*2*4*28 = 512)."""
    for H, C, Hs, MT in ((8, 2, 4, 1), (128, 8, 16, 1), (144, 8, 20, 2), (224, 8, 28, 2)):
        p = plan("GRU", H, 32, True)
        assert (p["family"], p["C"], p["Hs"], p["MT"]) == ("tc_cluster", C, Hs, MT), H
        assert H - (C - 1) * Hs > 0
    assert plan("GRU", 228, 32, False)["family"] == "ffma"


def test_persistent_slicing_at_b200_parameters(clean_env):
    p = plan("GRU", 512, 300, False)
    assert (p["BT"], p["tiles_per_launch"], p["launches"], p["C"], p["Hs"]) == (128, 2, 2, 64, 8)
    p = plan("GRU", 512, 300, True)
    assert (p["BT"], p["splitk"], p["tiles_per_launch"], p["launches"], p["C"], p["Hs"]) == (32, 1, 9, 2, 4, 128)
    clean_env.setenv("SBR_DISABLE_SPLITK_SCAN", "1")
    p = plan("GRU", 512, 1200, True)
    assert (p["splitk"], p["tiles_per_launch"], p["launches"]) == (0, 37, 2)
    assert plan("GRU", 512, 1184, True)["launches"] == 1


def test_argument_errors(clean_env):
    from sbr_b200 import _capi
    assert plan("GRU", 513, 32, False) is None          # no scan holds H > 512
    assert plan("GRU", 0, 32, False) is None
    clean_env.setenv("SBR_SCAN_MULTICAST", "1")
    assert plan("GRU", 512, 32, False) is None          # not modelled
    out = _capi.SbrScanPlan()
    lib = _capi.load_library()
    assert lib.sbr_plan_layer_scan(None, 1, 64, 32, None, 10, 0, 148, None, 37, out) == -1   # no device description


def _compiled_variants():
    """Template cases of the dispatch code, read from the sources."""
    src = {f: open(os.path.join(CSRC, f)).read() for f in ("rnn_tc.cu", "rnn_cluster.cu", "tc_scan.cu", "tc_gemm.cu")}
    out = set()
    s = src["rnn_tc.cu"]
    for G, BT in re.findall(r"SBR_FWD_CASE\((\d), (\d+)\)", s):
        out.add(("tc", "fwd", int(G), int(BT)))
    body = s[s.index("#define SBR_BWD_CASE"):]
    body = body[:body.index("#undef SBR_BWD_CASE")]
    bts = [int(b) for b in re.findall(r"rnn_bwd_tc_kernel<G_, MT_, (\d+)>", body)]
    assert sorted(bts) == [8, 16]
    for G, MT in re.findall(r"SBR_BWD_CASE\((\d), (\d)\)", body):
        for bt in bts:
            out.add(("tc", "bwd", int(G), int(MT), bt))
    for d, G, BT, JU, WS in re.findall(r"SBR_FFMA_(FWD|BWD)\((\d), (\d+), (\d), (true|false)\)", src["rnn_cluster.cu"]):
        out.add(("ffma", d.lower(), int(G), int(BT), int(JU), WS == "true"))
    s = src["tc_scan.cu"]
    for G in re.findall(r"launch_cluster_coop\(m, tc_scan_fwd_kernel<(\d)>", s):
        out.add(("persistent", "fwd", int(G), "launch"))
    for G in re.findall(r"launch_cluster_coop\(m, tc_scan_bwd2_kernel<(\d)>", s):
        out.add(("persistent", "bwd", int(G), "splitk"))
    for G in re.findall(r"launch_coop\(m, tc_scan_bwd_kernel<(\d)>", s):
        out.add(("persistent", "bwd", int(G), "nosplit"))
    cells = {"LSTM": 4, "GRU": 3, "VAN": 1}
    for c, d in re.findall(r"launch_tg<EPI_(LSTM|GRU|VAN)_(FWD|BWD)>", src["tc_gemm.cu"]):
        out.add(("step", d.lower(), cells[c]))
    return out


# switch settings a user can run with; the FFMA scans are reached for every H once the tensor-core scans are off
ENVS = [{}, {"SBR_TC_BT": "8"}, {"SBR_TC_BT": "16"}, {"SBR_DISABLE_SPLITK_SCAN": "1"}, {"SBR_DISABLE_PERSISTENT_SCAN": "1"},
        {"SBR_DISABLE_TC_BWD": "1"}, {"SBR_DISABLE_TC": "1", "SBR_DISABLE_STEP_SCAN": "1"}]
# batch sizes on both sides of every one-wave threshold of the FFMA tile choice (cdiv(B, BT) * C <= 148)
FFMA_BS = sorted({1, 5000} | {bt * (148 // c) + d for bt in (8, 16, 32) for c in (1, 2, 4, 8) for d in (0, 1)})
OTHER_BS = [1, 32, 300, 1200, 5000]


def _reachable(monkeypatch):
    out = set()
    for env in ENVS:
        for k in SWITCHES:
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        Bs = FFMA_BS if "SBR_DISABLE_STEP_SCAN" in env else OTHER_BS
        for cell in ("LSTM", "GRU", "Vanilla"):
            for H in range(1, 513):
                for B in Bs:
                    for backward in (False, True):
                        out.add(variant(plan(cell, H, B, backward), backward))
    return out


@pytest.fixture(scope="module")
def reachable():
    mp = pytest.MonkeyPatch()
    try:
        return _reachable(mp)
    finally:
        mp.undo()


def test_every_compiled_variant_is_reachable_and_every_reachable_one_compiled(reachable):
    compiled = _compiled_variants()
    assert len([v for v in compiled if v[0] == "ffma"]) == 37
    assert not compiled - reachable, "compiled but never selected: %s" % sorted(compiled - reachable)
    assert not reachable - compiled, "selected without a kernel: %s" % sorted(reachable - compiled)


def _case_plans(case):
    import zlib
    import numpy as np
    from tests.test_gpu_parity import _init
    from oracle import sbr_oracle as O
    spec = O.Spec(n_items=97, cell=case["cell"], layers=case["layers"], loss="CCE")
    rng, _ = _init(spec, zlib.crc32(case["id"].encode()))
    _, _, lens = scan_batch(rng, case["B"], case["T"], 97)
    assert lens.max() == case["T"] and lens.min() == 1 and len(set(lens.tolist())) > 2
    return [(plan(case["cell"], H, case["B"], False, lens, case["T"]), plan(case["cell"], H, case["B"], True, lens, case["T"]))
            for H in case["layers"]]


@pytest.mark.parametrize("case", CASES, ids=[c["id"] for c in CASES])
def test_gpu_case_plans_to_its_variant(case, clean_env):
    for k, v in case["env"].items():
        clean_env.setenv(k, v)
    plans = _case_plans(case)
    assert [(variant(f, False), variant(b, True)) for f, b in plans] == case["expect"]
    if case["sliced"]:
        assert all(p["launches"] >= 2 for p in plans[-1])
    assert case["T"] >= 9


def test_gpu_cases_cover_every_reachable_variant(reachable):
    covered = {v for c in CASES for pair in c["expect"] for v in pair}
    assert not reachable - covered, "no GPU case runs: %s" % sorted(reachable - covered)
    assert len({c["id"] for c in CASES}) == len(CASES)
