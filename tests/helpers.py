"""Shared helpers for the parity tests (test infrastructure)."""
import hashlib
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def load_golden():
    with open(os.path.join(HERE, "golden", "golden.json")) as f:
        return json.load(f)


def load_reference_cases():
    with open(os.path.join(HERE, "golden", "reference_cases.json")) as f:
        return json.load(f)


def golden_payload(seed, nrows, disp, dtype):
    """Same recipe as tests/golden/make_golden.py::payload (raw random bytes -> NaNs, -0, denormals...)."""
    rng = np.random.default_rng(seed)
    raw = rng.integers(0, 256, size=nrows * disp * np.dtype(dtype).itemsize, dtype=np.uint8)
    return raw.view(dtype).reshape(nrows, disp)


def golden_world_shards(w):
    return [golden_payload(w["seed"] + r, w["nrows"][r], w["disp"], w["dtype"]) for r in range(len(w["nrows"]))]


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def random_world(rng, P, dtype, disp, max_rows=200, allow_empty=True):
    nrows = [int(rng.integers(0 if allow_empty else 1, max_rows)) for _ in range(P)]
    if sum(nrows) == 0:
        nrows[-1] = 5
    shards = []
    for n in nrows:
        raw = rng.integers(0, 256, size=n * disp * np.dtype(dtype).itemsize, dtype=np.uint8)
        shards.append(raw.view(dtype).reshape(n, disp))
    return nrows, shards


def random_valid_requests(rng, lenlist, B, max_count=40):
    """Requests that never straddle an owner (include/ddstore.hpp:213-214)."""
    bounds = [0] + [int(x) for x in lenlist]
    owners = [r for r in range(len(lenlist)) if bounds[r + 1] > bounds[r]]
    starts, counts = [], []
    for _ in range(B):
        r = owners[int(rng.integers(0, len(owners)))]
        lo, hi = bounds[r], bounds[r + 1]
        s = int(rng.integers(lo, hi))
        c = int(rng.integers(0, min(max_count, hi - s) + 1))
        starts.append(s)
        counts.append(c)
    return np.array(starts, np.int64), np.array(counts, np.int64)
