"""The oracle is pinned here: C restatement (oracle/ddstore_oracle.c) and NumPy restatement
(oracle/oracle.py) against
  (1) the committed golden vectors the unmodified reference produced (tests/golden/golden.json),
  (2) the reference's own known answers (test/demo.cxx:20-37, test/demo.py:55-56, test/test.py:157-159),
  (3) what the verbatim-compiled reference (oracle/_ref) returned on seeded random worlds
      (tests/golden/reference_cases.json).
CPU only."""
import hashlib

import numpy as np
import pytest

from oracle import oracle as O
from tests.helpers import (golden_world_shards, load_golden, load_reference_cases, random_valid_requests, random_world,
                           sha)

G = load_golden()
R = load_reference_cases()


def test_sortedsearch_golden(coracle):
    for case in G["sortedsearch"]:
        for num, tgt in zip(case["nums"], case["targets"]):
            assert coracle.sortedsearch(case["lenlist"], num) == tgt
            assert O.np_sortedsearch(case["lenlist"], num) == tgt


def test_sortedsearch_survey_tables(coracle):
    # SURVEY.md section 4, [probe] tables
    ll = [4, 8, 12, 16]
    exp = {-1: 0, 0: 0, 3: 0, 4: 1, 7: 1, 8: 2, 11: 2, 12: 3, 15: 3, 16: 0, 17: 0}
    for k, v in exp.items():
        assert coracle.sortedsearch(ll, k) == v
    assert [coracle.sortedsearch([0, 5, 5, 9], n) for n in range(0, 10)] == [1] * 5 + [3] * 4 + [0]
    assert [coracle.sortedsearch([0, 0, 7], n) for n in range(0, 8)] == [2] * 7 + [0]
    assert all(coracle.sortedsearch([5, 5, 5], n) == 0 for n in range(-1, 8))


@pytest.mark.parametrize("w", G["worlds"], ids=[w["name"] for w in G["worlds"]])
def test_worlds_golden(coracle, w):
    shards = golden_world_shards(w)
    ll, rc = coracle.lenlist(w["nrows"], [w["disp"]] * len(w["nrows"]))
    assert rc == 0 and ll.tolist() == w["lenlist"] == O.np_lenlist(w["nrows"]).tolist()
    good = []
    for r in w["requests"]:
        for impl in (coracle.get_batch, O.np_get_batch):
            out, offs, bad, rc = impl(shards, [r["start"]], [r["count"]])
            if "error" in r:
                assert bad == 0 and O.ERR_TEXT[rc] == r["error"]
            else:
                assert bad == -1 and rc == 0
                assert sha(out.tobytes()) == r["sha256"]
                if "hex" in r:
                    assert out.tobytes().hex() == r["hex"]
        if "error" not in r:
            good.append((r["start"], r["count"]))
    for impl in (coracle.get_batch, O.np_get_batch):
        out, offs, bad, rc = impl(shards, [g[0] for g in good], [g[1] for g in good])
        assert bad == -1 and out.size == w["batch_nbytes"] and sha(out.tobytes()) == w["batch_sha256"]
        row = w["disp"] * w["itemsize"]
        assert offs.tolist() == np.concatenate([[0], np.cumsum([g[1] * row for g in good])]).tolist()


def test_batch_stops_at_first_bad(coracle):
    w = G["worlds"][0]
    shards = golden_world_shards(w)
    starts = [r["start"] for r in w["requests"]]
    counts = [r["count"] for r in w["requests"]]
    first_bad = next(i for i, r in enumerate(w["requests"]) if "error" in r)
    for impl in (coracle.get_batch, O.np_get_batch):
        out, offs, bad, rc = impl(shards, starts, counts)
        assert bad == first_bad and O.ERR_TEXT[rc] == w["requests"][first_bad]["error"]
        assert out.size == sum(c for c in counts[:first_bad]) * w["disp"] * w["itemsize"]


def test_demo_cxx_known_answer(coracle):
    # test/demo.cxx:20-37 at P=2: rank0 reads row 3 = {13,14}; rank1 reads row 1 = {3,4}
    shards = [np.array([1, 2, 3, 4], np.float64).reshape(2, 2) + 10 * r for r in range(2)]
    for rec in G["demo_cxx"]:
        out, _, bad, rc = coracle.get_batch(shards, [rec["start"]], [1])
        assert bad == -1 and out.view(np.float64).tolist() == rec["got"]
    assert G["demo_cxx"][0]["got"] == [13.0, 14.0] and G["demo_cxx"][1]["got"] == [3.0, 4.0]


@pytest.mark.parametrize("dt", ["float64", "float32"])
def test_demo_py_mean_property(coracle, dt):
    # test/demo.py:37,55-56 and test/test.py:157-159: shard r is all (r+1); mean(row idx) == idx//num + 1
    rec = G["demo_py"][dt]
    shards = [np.ones((rec["num"], rec["dim"]), dt) * (r + 1) for r in range(rec["P"])]
    for idx, mean in zip(rec["idx"], rec["means"]):
        out, _, bad, rc = coracle.get_batch(shards, [idx], [1])
        assert bad == -1
        assert float(np.mean(out.view(dt))) == mean == idx // rec["num"] + 1


def test_dtype_mismatch(coracle):
    shards = [np.zeros((4, 2), np.float32)]
    out, offs, bad, rc = coracle.get_batch(shards, [0], [1], req_itemsize=8)
    assert bad == 0 and O.ERR_TEXT[rc] == "Invalid data type"


def test_disp_mismatch(coracle):
    _, rc = coracle.lenlist([3, 3], [4, 5])
    assert O.ERR_TEXT[rc] == "Invalid disp"


def test_synth_generator_c_vs_numpy(coracle):
    for dt in (np.float32, np.int64, np.uint8, np.float64, np.int32):
        a = coracle.synth_rows(0xDD5, 1234567, 9, 13, dt)
        b = O.np_synth_rows(0xDD5, 1234567, 9, 13, dt)
        assert a.tobytes() == b.tobytes()
    f = coracle.synth_rows(0xDD5, 0, 4096, 64, np.float32)
    assert np.isnan(f).any()  # payload deliberately contains NaN bit patterns


@pytest.mark.parametrize("dtype,disp,P", [(np.float32, 1, 4), (np.float32, 16, 8), (np.int64, 2, 3),
                                          (np.uint8, 7, 2), (np.float64, 5, 1), (np.int32, 3, 5), (np.bool_, 3, 2)])
def test_c_oracle_vs_compiled_reference(coracle, dtype, disp, P):
    """against what the compiled reference returned on the same seeded world (tests/golden/reference_cases.json)"""
    ref = next(w for w in R["random_worlds"] if (w["dtype"], w["disp"], w["P"]) == (np.dtype(dtype).name, disp, P))
    rng = np.random.default_rng(1000 + disp * 31 + P)
    nrows, shards = random_world(rng, P, dtype, disp)
    ll = O.np_lenlist(nrows)
    assert nrows == ref["nrows"] and ll.tolist() == ref["lenlist"]
    assert ref["ref_disp"] == disp and ref["itemsize"] == np.dtype(dtype).itemsize
    starts, counts = random_valid_requests(rng, ll, 300)
    c_out, c_offs, cbad, rc = coracle.get_batch(shards, starts, counts)
    n_out, n_offs, nbad, nrc = O.np_get_batch(shards, starts, counts)
    assert cbad == nbad == -1
    assert c_out.size == ref["batch_nbytes"] and sha(c_out.tobytes()) == ref["batch_sha256"]
    assert c_out.tobytes() == n_out.tobytes()
    assert c_offs.tolist() == n_offs.tolist()
    # error classification agrees request by request on arbitrary (mostly invalid) requests
    total = int(ll[-1])
    rows = hashlib.sha256()
    for code in ref["probes"]:
        s = int(rng.integers(-5, total + 5))
        c = int(rng.integers(0, 60))
        t, off, rc = coracle.locate(ll, s, c)
        assert (O.ERR_TEXT[rc] if rc else None) == R["outcome_codes"][code]
        assert O.np_locate(ll, s, c)[2] == rc
        if not rc:
            o2, _, _, _ = coracle.get_batch(shards, [s], [c])
            rows.update(o2.tobytes())
    assert rows.hexdigest() == ref["probe_rows_sha256"]


def test_reference_init_update_and_fences(coracle):
    # include/ddstore.hpp:110-195 and src/ddstore.cxx:51-77: what the compiled reference returned, against the restatement
    ref = R["init_update_fences"]
    shards = [np.zeros((n, ref["disp"]), np.float32) for n in ref["nrows"]]
    a = np.array(ref["update"]["rows"], np.float32)
    u = ref["update"]["offset"]
    shards[ref["update"]["rank"]][u:u + len(a)] = a
    exp = np.zeros((4, 3), np.float32)
    exp[1:3] = np.arange(6, dtype=np.float32).reshape(2, 3)
    for impl in (coracle.get_batch, O.np_get_batch):
        out, _, bad, _ = impl(shards, [ref["get"]["start"]], [ref["get"]["count"]])
        assert bad == -1 and out.tobytes().hex() == ref["get"]["hex"] == exp.tobytes().hex()
    assert ref["errors"] == {"epoch_begin_twice": "Fence already activated", "epoch_end_twice": "Fence is not activated",
                             "add_disp_3_4_3": "Invalid disp"}
    _, rc = coracle.lenlist([2, 2, 2], [3, 4, 3])
    assert O.ERR_TEXT[rc] == ref["errors"]["add_disp_3_4_3"]
