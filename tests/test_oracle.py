"""CPU tests: the C restatement (oracle/louvain_oracle.c) and our RGG generator are pinned against the
golden traces captured from the unmodified reference (tests/golden/ref_traces.json)."""
import os

import numpy as np
import pytest

from helpers import assert_trace_matches, case_graph
from oracle import oracle as O


def _names(golden_cases, prefix):
    return sorted(k for k in golden_cases if k.startswith(prefix))


def test_golden_file_has_all_kinds(golden):
    kinds = {c["kind"] for c in golden.values()}
    assert kinds == {"rgg", "file_rgg", "hand", "file_balanced"}
    assert golden["rgg_n16384_p1"]["modularity"] == "0.75671532450841406"   # SURVEY.md 8(c) known answer
    assert golden["rgg_n16384_p1"]["final_chash"] == "5bf1e47053c42601"
    # SURVEY.md 8(c), p-strip graphs made by the reference generator on p ranks, and the shard-combinable trace hashes
    for name, ne, iters, mod, ch in (("rgg_n16384_p2", 131178, 16, "0.77055664274182301", "80ae93c9830e0ce7"),
                                     ("rgg_n16384_p4", 129262, 14, "0.76142299956738535", "cd26d5284d897ead"),
                                     ("rgg_n16384_p8", 130920, 20, "0.74390133494621125", "2a8ec661d39110ca"),
                                     ("rgg_n65536_p1", 564602, 18, "0.76023592129323059", None)):
        c = golden[name]
        assert (c["ne"], c["iters"], c["modularity"]) == (ne, iters, mod), name
        assert ch is None or c["final_chash"] == ch, name
    tr = golden["rgg_n16384_p1"]["trace"]
    assert (tr[0]["modularity"], tr[0]["moved"], tr[0]["chash"]) == ("0.00017722880436126689", 9302, "6e0f20678d8ceb80")
    assert (tr[1]["modularity"], tr[1]["moved"], tr[1]["chash"]) == ("0.2003383411625265", 9028, "85e25e5c7dba5389")
    assert (tr[13]["moved"], tr[13]["chash"]) == (738, "e9f74809e145f6bd")          # the rejected 14th iteration
    # SURVEY.md 8(c): `miniVite -n 524288` on 1 and 8 ranks (graph files written by our byte-identical generator)
    c1, c8 = golden["file_rgg_n524288_s1_p1"], golden["file_rgg_n524288_s8_p8"]
    assert (c1["ne"], c1["iters"], c1["modularity"]) == (4997382, 20, "0.75810023251607561")
    assert (c8["ne"], c8["iters"], c8["modularity"]) == (5003290, 19, "0.75862461064860043")


def test_oracle_matches_every_golden_case(golden):
    for name, case in golden.items():
        parts, rps, eds, _keep = case_graph(case)
        assert sum(len(e) for e in eds) == case["ne"], name      # same graph as the reference built / read
        res = O.louvain(parts, rps, eds)
        comm = np.concatenate(res["comm"])
        assert_trace_matches(case, res["iters"], res["modularity"], res["trace"], res["chash_final"], comm)
        assert repr(res["constant"]) == case["constant"], name


def test_partition_invariance_unit_weights(golden):
    """Same global graph on 1/2/4/8 shards -> identical traces (SURVEY.md 8(e))."""
    base = golden["file_rgg_n16384_s4_p1"]
    for p in (2, 4, 8):
        c = golden[f"file_rgg_n16384_s4_p{p}"]
        assert c["trace"] == base["trace"] and c["modularity"] == base["modularity"]


def test_first_iteration_rejected_returns_lower():
    """dspl.hpp:1401-1440: if iteration 1 fails the test the function returns `lower` with iters == 1."""
    # a graph without edges: modularity 0 - (-1) >= thresh, so use lower = 0.5 to force rejection
    parts = np.array([0, 4], np.int64)
    rp = np.array([0, 1, 2, 3, 4], np.int64)
    ed = np.zeros(4, O.EDGE_DTYPE)
    ed["tail"] = [1, 0, 3, 2]
    ed["weight"] = 1.0
    res = O.louvain(parts, [rp], [ed], lower=0.9)
    assert res["iters"] == 1 and res["modularity"] == 0.9
    assert list(res["comm"][0]) == [0, 1, 2, 3]


def test_oracle_against_live_reference():
    """The reference's own run (`-f` on 2 ranks) of the 2-strip RGG with 8192 vertices, as it reported it
    (tests/golden/make_golden_oracle_check.py)."""
    import json
    from minivite_b200 import hostgraph as hg
    with open(os.path.join(os.path.dirname(__file__), "golden", "oracle_check_n8192_s2.json")) as f:
        ref = json.load(f)
    ss = hg.generate_rgg(ref["n"], ref["strips"])
    res = O.louvain(ss.shards[0].parts, [s.rowptr for s in ss.shards], [s.edges for s in ss.shards])
    assert res["iters"] == ref["iters"] and res["modularity"] == float(ref["modularity"])
    assert [int(t["chash"]) for t in res["trace"]] == [int(h, 16) for h in ref["chash"]]


def test_balanced_reader_matches_reference_bins(golden, tmp_path):
    """BinaryEdgeList::read_balanced (-b): same vertex bins as the reference's greedy edge balancing (graph.hpp:416-461)."""
    from minivite_b200 import hostgraph as hg
    case = golden["file_balanced_n16384_p4"]
    ss = hg.generate_rgg(case["n"], 1, random_edge_percent=case["pct"])
    path = str(tmp_path / "g.bin")
    ss.write(path)
    for r in range(4):
        sh = hg.read_graph(path, r, 4, balanced=True).shards[0]
        assert list(sh.parts) == case["parts"]
        assert sh.base == case["parts"][r] and sh.lnv == case["parts"][r + 1] - case["parts"][r]
    # vertex-balanced reader for comparison
    sh = hg.read_graph(path, 1, 4, balanced=False).shards[0]
    assert sh.base == 4096 and sh.lnv == 4096


def _fnv1a_words(vec):
    h = 1469598103934665603
    for v in vec.tolist():
        h = ((h ^ (v & 0xFFFFFFFFFFFFFFFF)) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return "%016x" % h


@pytest.mark.parametrize("name,ncomm,fnv", [("rgg_n16384_p1", 1953, "2788b5ffe2f49136"),
                                            ("rgg_n65536_p1", 6889, "3cf802502bc50070"),
                                            ("file_rgg_n524288_s1_p1", 48778, "188df44bd1f5b787")])
def test_final_assignment_matches_survey_known_answers(golden, name, ncomm, fnv):
    """SURVEY.md 8(c): number of communities and FNV-1a hash of the final currComm, captured from the unmodified
    reference in a separate probe session (a pin that does not pass through this repo's own hash or hooks)."""
    parts, rps, eds, _keep = case_graph(golden[name])
    res = O.louvain(parts, rps, eds)
    comm = np.concatenate(res["comm"])
    assert len(np.unique(comm)) == ncomm
    assert _fnv1a_words(comm) == fnv


def test_rgg_radius_matches_survey_table():
    from minivite_b200 import hostgraph as hg
    assert abs(hg.rgg_radius(16384) - 1.249e-2) < 5e-6          # SURVEY.md section 8 config table (graph.hpp:629-631)
    assert abs(hg.rgg_radius(16777216) - 4.567e-4) < 5e-8
    assert abs(hg.rgg_radius(67108864, 8) - 2.341e-4) < 5e-8


def test_oracle_matches_power_law_goldens(golden_rmat):
    """R-MAT graphs (hubs of degree 3 684 and 15 706), plain and edge-balanced (-b) splits: the C restatement
    reproduces the unmodified reference's traces bit for bit."""
    from helpers import assert_trace_matches, case_graph
    from oracle import oracle as O
    for name, case in golden_rmat.items():
        parts, rps, eds, _ = case_graph(case)
        r = O.louvain(parts, rps, eds)
        tr = [{"modularity": t["modularity"], "moved": t["moved"], "chash": t["chash"]} for t in r["trace"]]
        assert_trace_matches(case, r["iters"], r["modularity"], tr, r["chash_final"])
        assert repr(r["constant"]) == case["constant"], name
