"""tests/golden/make_golden.py -- generates tests/golden/golden.json and tests/golden/reference_cases.json.

Runs the UNMODIFIED reference (oracle/_ref/libddstore_ref.so: /root/reference/include/ddstore.hpp
+ src/ddstore.cxx compiled verbatim against oracle/mpi_shim) on small seeded worlds and records,
for every case, the inputs (as a recipe) and what the reference wrote (hex for small outputs,
sha256 otherwise). Needs /root/reference, so it runs in the build container only; the JSON it
writes is committed and is what travels to the GPU box.

    python tests/golden/make_golden.py
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.oracle import RefWorld  # noqa: E402
from tests.helpers import random_valid_requests, random_world  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden.json")
OUT_REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_cases.json")


def payload(seed, nrows, disp, dtype):
    """Deterministic shard contents incl. NaN / -0 / denormal / negative patterns: raw random bytes."""
    rng = np.random.default_rng(seed)
    raw = rng.integers(0, 256, size=nrows * disp * np.dtype(dtype).itemsize, dtype=np.uint8)
    return raw.view(dtype).reshape(nrows, disp)


def case_sortedsearch(w):
    out = []
    for ll in ([4, 8, 12, 16], [0, 5, 5, 9], [0, 0, 7], [5, 5, 5], [7], [3, 3, 10, 10, 12]):
        nums = list(range(-2, ll[-1] + 3))
        out.append({"lenlist": ll, "nums": nums, "targets": [w.sortedsearch(ll, n) for n in nums]})
    return out


def case_world(name, seed, nrows, disp, dtype, requests, rank):
    """requests: list of (start, count). Records per-request outcome of get() as rank `rank`."""
    P = len(nrows)
    w = RefWorld(P)
    shards = [payload(seed + r, nrows[r], disp, dtype) for r in range(P)]
    w.add("v", shards)
    it, dp, ll = w.query(rank, "v")
    rec = {"name": name, "seed": seed, "nrows": nrows, "disp": disp, "dtype": np.dtype(dtype).name, "rank": rank,
           "itemsize": it, "ref_disp": dp, "lenlist": ll.tolist(), "requests": []}
    for (st, ct) in requests:
        buf = np.zeros((max(ct, 0), disp), dtype)
        try:
            w.get(rank, "v", buf, st)
            b = buf.tobytes()
            r = {"start": st, "count": ct, "sha256": hashlib.sha256(b).hexdigest()}
            if len(b) <= 64:
                r["hex"] = b.hex()
        except ValueError as e:
            r = {"start": st, "count": ct, "error": str(e)}
        rec["requests"].append(r)
    # the batched view: serial loop over the valid requests only
    good = [(s, c) for (s, c), r in zip(requests, rec["requests"]) if "error" not in r]
    packed, bad, err, _ = w.get_batch(rank, "v", [g[0] for g in good], [g[1] for g in good])
    assert bad == -1 and err is None
    rec["batch_sha256"] = hashlib.sha256(packed.tobytes()).hexdigest()
    rec["batch_nbytes"] = int(packed.size)
    w.close()
    return rec


def case_demo_cxx():
    """test/demo.cxx:20-37 with P=2 (method 0 instead of the hard-coded libfabric method)."""
    w = RefWorld(2)
    shards = [np.array([1, 2, 3, 4], np.float64).reshape(2, 2) + 10 * r for r in range(2)]
    w.add("var", shards)
    res = []
    for rank in range(2):
        getbuf = np.zeros((1, 2), np.float64)
        start = (2 * (rank + 1)) % (2 * 2) + 1
        w.get(rank, "var", getbuf, start)
        res.append({"rank": rank, "start": start, "got": getbuf.reshape(-1).tolist()})
    w.close()
    return res


def case_demo_py(seed=20260921):
    """test/demo.py:35-56 and test/test.py:144-159 shape: shard r == r+1, single-row gets, mean check.
    Scaled to num=4096 rows (the mean property does not depend on num)."""
    P, num, dim = 2, 4096, 64
    out = {}
    for dt in ("float64", "float32"):
        w = RefWorld(P)
        w.add("var", [np.ones((num, dim), dt) * (r + 1) for r in range(P)])
        rng = np.random.default_rng(seed)
        idxs = rng.integers(0, num * P, size=32).tolist()
        means = []
        for idx in idxs:
            buff = np.zeros((1, dim), dt)
            w.epoch_begin()
            w.get(1, "var", buff, idx)
            w.epoch_end()
            means.append(float(np.mean(buff)))
            assert means[-1] == idx // num + 1
        out[dt] = {"P": P, "num": num, "dim": dim, "idx": idxs, "means": means}
        w.close()
    return out


RANDOM_WORLDS = [("float32", 1, 4), ("float32", 16, 8), ("int64", 2, 3), ("uint8", 7, 2), ("float64", 5, 1),
                 ("int32", 3, 5), ("bool", 3, 2)]
OUTCOME_CODES = {None: ".", "Invalid start on target": "s", "Invalid count on target": "c"}


def case_random_world(dtype, disp, P):
    """a seeded random world, 300 valid requests as one serial get() loop, then 400 arbitrary (mostly invalid) single
    get() calls: their outcome (one letter of OUTCOME_CODES each) and the sha256 of the rows of the valid ones, in order"""
    dt = np.dtype(dtype)
    seed = 1000 + disp * 31 + P
    rng = np.random.default_rng(seed)
    nrows, shards = random_world(rng, P, dt, disp)
    w = RefWorld(P)
    w.add("v", shards)
    it, dp, ll = w.query(0, "v")
    starts, counts = random_valid_requests(rng, ll, 300)
    out, bad, err, _ = w.get_batch(P - 1, "v", starts, counts)
    assert bad == -1 and err is None
    rec = {"dtype": dt.name, "disp": disp, "P": P, "seed": seed, "nrows": nrows, "itemsize": it, "ref_disp": dp,
           "lenlist": ll.tolist(), "batch_nbytes": int(out.size), "batch_sha256": hashlib.sha256(out.tobytes()).hexdigest()}
    total = int(ll[-1])
    codes, h = [], hashlib.sha256()
    for _ in range(400):
        s = int(rng.integers(-5, total + 5))
        c = int(rng.integers(0, 60))
        buf = np.zeros((c, disp), dt)
        try:
            w.get(0, "v", buf, s)
            codes.append(OUTCOME_CODES[None])
            h.update(buf.tobytes())
        except ValueError as e:
            codes.append(OUTCOME_CODES[str(e)])
    rec["probes"] = "".join(codes)
    rec["probe_rows_sha256"] = h.hexdigest()
    w.close()
    return rec


def case_init_update_fences():
    """include/ddstore.hpp:110-195 and src/ddstore.cxx:51-77: init over 3 ranks (one empty), update 2 rows of rank 0
    at row offset 1, read the first 4 global rows from rank 2; then the fence and disp errors"""
    w = RefWorld(3)
    w.init("z", [4, 0, 6], [3, 3, 3], 4, np.float32)
    a = np.arange(6, dtype=np.float32).reshape(2, 3)
    w.update(0, "z", a, 1)
    got = np.full((4, 3), -1, np.float32)
    w.get(2, "z", got, 0)
    rec = {"P": 3, "nrows": [4, 0, 6], "disp": 3, "update": {"rank": 0, "offset": 1, "rows": a.tolist()},
           "get": {"rank": 2, "start": 0, "count": 4, "hex": got.tobytes().hex()}, "errors": {}}
    w.epoch_begin()
    for key, fn, exc in (("epoch_begin_twice", w.epoch_begin, RuntimeError), ("epoch_end", w.epoch_end, None),
                         ("epoch_end_twice", w.epoch_end, RuntimeError),
                         ("add_disp_3_4_3", lambda: w.add("bad", [np.zeros((2, d), np.float32) for d in (3, 4, 3)]),
                          ValueError)):
        try:
            fn()
            assert exc is None, key
        except (RuntimeError, ValueError) as e:
            assert isinstance(e, exc), key
            rec["errors"][key] = str(e)
    w.close()
    return rec


def case_owner_lookup(n=500):
    """src/ddstore.cxx:5-17 on seeded random row counts (1..12 ranks, 0..40 rows each, also empty ranks) and starts
    in [-5, 500]: [nrows, start, owner]"""
    w = RefWorld(1)
    rng = np.random.default_rng(11)
    out = []
    for _ in range(n):
        nrows = rng.integers(0, 41, size=int(rng.integers(1, 13))).tolist()
        start = int(rng.integers(-5, 501))
        out.append([nrows, start, w.sortedsearch(np.cumsum(nrows), start)])
    w.close()
    return out


def write_reference_cases():
    g = {"generator": "tests/golden/make_golden.py over oracle/_ref/libddstore_ref.so (reference @ 9035c779)",
         "outcome_codes": {v: k for k, v in OUTCOME_CODES.items()},
         "random_worlds": [case_random_world(*c) for c in RANDOM_WORLDS],
         "init_update_fences": case_init_update_fences(),
         "owner_lookup": case_owner_lookup()}
    # one top-level entry (or list element) per line: small enough to review, still plain JSON
    parts = []
    for k, v in g.items():
        if isinstance(v, list):
            body = "[\n  " + ",\n  ".join(json.dumps(x, separators=(",", ":")) for x in v) + "\n ]"
        else:
            body = json.dumps(v, separators=(",", ":"))
        parts.append(f" {json.dumps(k)}: {body}")
    with open(OUT_REF, "w") as f:
        f.write("{\n" + ",\n".join(parts) + "\n}\n")
    print("wrote", OUT_REF, os.path.getsize(OUT_REF), "bytes")


def main():
    write_reference_cases()
    w = RefWorld(1)
    g = {"generator": "tests/golden/make_golden.py over oracle/_ref/libddstore_ref.so (reference @ 9035c779)",
         "sortedsearch": case_sortedsearch(w)}
    w.close()
    rng = np.random.default_rng(7)
    worlds = []
    # fixed-stride float32, 4 ranks, incl. errors: negative start, straddle, past the end, count 0
    reqs = [(int(s), 1) for s in rng.integers(0, 4 * 50, size=24)] + \
           [(-1, 1), (49, 2), (200, 1), (199, 2), (0, 0), (50, 0), (10, 40), (150, 50), (0, 51), (200, 0)]
    worlds.append(case_world("fixed_f32_p4", 100, [50, 50, 50, 50], 16, np.float32, reqs, 2))
    # variable-length rows of disp=1 float32 (cfg3 shape), ranks of unequal size, one empty rank
    reqs = [(0, 100), (100, 1), (101, 899), (1000, 1), (1000, 2500), (3499, 1), (3500, 777), (4277, 5723),
            (9999, 1), (10000, 1), (999, 2), (3400, 101), (5, 3), (7, 1)]
    worlds.append(case_world("varlen_f32_p4_empty_rank", 200, [1000, 2500, 0, 6500], 1, np.float32, reqs, 0))
    # int64 disp=2 (edge_index shape), P=3
    reqs = [(int(s), int(c)) for s, c in zip(rng.integers(0, 300, size=20), rng.integers(1, 30, size=20))]
    worlds.append(case_world("edges_i64_p3", 300, [100, 120, 80], 2, np.int64, reqs, 1))
    # uint8 odd disp (byte-granular misalignment), P=2
    reqs = [(int(s), int(c)) for s, c in zip(rng.integers(0, 400, size=20), rng.integers(1, 9, size=20))]
    worlds.append(case_world("bytes_u8_p2", 400, [211, 189], 7, np.uint8, reqs, 1))
    # float64 P=1
    reqs = [(0, 1), (63, 1), (10, 20), (0, 64), (64, 1), (60, 5)]
    worlds.append(case_world("f64_p1", 500, [64], 5, np.float64, reqs, 0))
    g["worlds"] = worlds
    g["demo_cxx"] = case_demo_cxx()
    g["demo_py"] = case_demo_py()
    with open(OUT, "w") as f:
        json.dump(g, f, indent=1)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
