"""CPU-only checks of the boundary: the C-ABI library loads and exports every symbol the header declares,
the host-side index math matches the oracle and the golden vectors, the communicators work across
threads / processes / a gloo process group (world_size 2), and the data plane FAILS LOUDLY without a GPU."""
import multiprocessing as mp
import os
import re
import subprocess
import sys
import threading
import uuid

import numpy as np
import pytest

from ddstore_b200 import _capi
from tests.helpers import load_golden, load_reference_cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = load_golden()


def _header_functions():
    src = open(os.path.join(ROOT, "include", "ddstore_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"\b(dds_[a-z_0-9]+)\s*\(", src)
    return sorted(set(n for n in names if not n.endswith("_fn")))


def test_library_exports_every_declared_symbol():
    L = _capi.lib()
    declared = _header_functions()
    assert len(declared) >= 28
    for name in declared:
        assert hasattr(L, name), f"{name} declared in include/ddstore_b200.h but not exported"
    assert sorted(_capi.SIGNATURES) == declared, "ctypes signature table and header diverged"
    out = subprocess.run(["nm", "-D", "--defined-only", _capi.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (dds_[a-z_0-9]+)", out))
    assert set(declared) <= exported


def test_strerror_carries_reference_texts():
    L = _capi.lib()
    exp = {1: "Invalid data type", 2: "Invalid start on target", 3: "Invalid count on target", 4: "Invalid disp",
           5: "Fence already activated", 6: "Fence is not activated"}
    for code, text in exp.items():
        assert L.dds_strerror(code).decode() == text


def _ss(ll, num):
    a = np.ascontiguousarray(ll, dtype=np.int64)
    return _capi.lib().dds_sortedsearch(a.ctypes.data_as(_capi.I64P), len(a), num)


def _locate(ll, start, count):
    import ctypes as C
    a = np.ascontiguousarray(ll, dtype=np.int64)
    owner, off = C.c_int(), C.c_int64()
    rc = _capi.lib().dds_locate(a.ctypes.data_as(_capi.I64P), len(a), start, count, C.byref(owner), C.byref(off))
    return owner.value, off.value, rc


def test_host_sortedsearch_golden():
    for case in G["sortedsearch"]:
        for num, tgt in zip(case["nums"], case["targets"]):
            assert _ss(case["lenlist"], num) == tgt


def test_host_locate_vs_oracle(coracle):
    rng = np.random.default_rng(5)
    for _ in range(200):
        P = int(rng.integers(1, 9))
        ll = np.cumsum(rng.integers(0, 50, size=P))
        for _ in range(50):
            s, c = int(rng.integers(-3, ll[-1] + 4)), int(rng.integers(0, 30))
            t, off, rc = coracle.locate(ll, s, c)
            assert _locate(ll, s, c) == (t, off, rc)
            if rc:
                assert _capi.last_error() == {2: "Invalid start on target", 3: "Invalid count on target"}[rc]


def test_golden_request_errors_host_side():
    for w in G["worlds"]:
        for r in w["requests"]:
            _, _, rc = _locate(w["lenlist"], r["start"], r["count"])
            assert (rc != 0) == ("error" in r)
            if rc:
                assert _capi.last_error() == r["error"]


def _thread_world(P, fn):
    key = "t" + uuid.uuid4().hex[:12]
    res, errs = [None] * P, []

    def run(r):
        try:
            from ddstore_b200.comm import ShmComm
            c = ShmComm(key, r, P)
            try:
                res[r] = fn(c, r)
            finally:
                c.close()
        except Exception as e:  # noqa: BLE001
            errs.append((r, repr(e)))

    th = [threading.Thread(target=run, args=(r,)) for r in range(P)]
    [t.start() for t in th]
    [t.join(60) for t in th]
    assert not errs, errs
    return res


def _exchange(c, nrows, disp):
    out = np.zeros(c.Get_size(), np.int64)
    rc = _capi.lib().dds_exchange_lenlist(c.handle, nrows, disp, out.ctypes.data_as(_capi.I64P))
    return rc, out.tolist()


def test_shm_comm_threads_allgather_barrier_lenlist():
    P = 4
    nrows = [1000, 2500, 0, 6500]

    def body(c, r):
        parts = c.allgather_bytes(bytes([r]) * 5000)  # > one 4 KiB slot: exercises the piecewise path
        assert parts == [bytes([i]) * 5000 for i in range(P)]
        for _ in range(20):
            c.Barrier()
        return _exchange(c, nrows[r], 3)

    for rc, ll in _thread_world(P, body):
        assert rc == 0 and ll == [1000, 3500, 3500, 10000]  # include/ddstore.hpp:84-89


def test_comm_split_builds_the_reference_replica_groups():
    """comm.Split(rank // width, rank) as in examples/vae/distdataset.py:28: consecutive ranks in groups of `width`,
    each group with its own rank numbering, allgather and lenlist"""
    P, width = 6, 2

    def body(c, r):
        sub = c.Split(r // width, r)
        try:
            assert sub.Get_size() == width and sub.Get_rank() == r % width
            parts = sub.allgather_bytes(bytes([r]))
            sub.Barrier()
            return [p[0] for p in parts], _exchange(sub, 10 * (r + 1), 2)
        finally:
            sub.close()

    res = _thread_world(P, body)
    for r, (members, (rc, ll)) in enumerate(res):
        g = r // width
        assert members == [g * width, g * width + 1] and rc == 0
        assert ll == [10 * (g * width + 1), 10 * (g * width + 1) + 10 * (g * width + 2)]
    # an uneven split (key reverses the order inside the colour)
    res = _thread_world(5, lambda c, r: (lambda s: (s.Get_rank(), s.Get_size(), s.close())[:2])(c.Split(r % 2, -r)))
    assert res == [(2, 3), (1, 2), (1, 3), (0, 2), (0, 3)]


def test_lenlist_disp_mismatch_raises_on_the_differing_ranks():
    # include/ddstore.hpp:78-82: ranks whose disp != max(disp) throw "Invalid disp"
    def body(c, r):
        rc, _ = _exchange(c, 10, 4 if r != 1 else 3)
        return rc, _capi.last_error()

    res = _thread_world(3, body)
    assert [r[0] for r in res] == [0, _capi.ERR_DISP, 0]
    assert res[1][1] == "Invalid disp"


def _proc_body(key, r, P, q):
    try:
        from ddstore_b200.comm import ShmComm
        c = ShmComm(key, r, P)
        parts = c.allgather_bytes(f"rank{r}".encode())
        c.Barrier()
        rc, ll = _exchange(c, 10 * (r + 1), 2)
        c.close()
        q.put((r, parts, rc, ll))
    except Exception as e:  # noqa: BLE001
        q.put((r, repr(e), -1, None))


def test_shm_comm_across_processes():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    key = "p" + uuid.uuid4().hex[:12]
    P = 2
    ps = [ctx.Process(target=_proc_body, args=(key, r, P, q)) for r in range(P)]
    [p.start() for p in ps]
    got = sorted(q.get(timeout=120) for _ in range(P))
    [p.join(30) for p in ps]
    for r, parts, rc, ll in got:
        assert parts == [b"rank0", b"rank1"] and rc == 0 and ll == [10, 30]


GLOO_SCRIPT = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch.distributed as dist
from ddstore_b200 import _capi
from ddstore_b200.comm import TorchDistComm
dist.init_process_group("gloo", init_method="env://")
c = TorchDistComm()
r, P = c.Get_rank(), c.Get_size()
assert c.allgather_bytes(bytes([65 + r]) * 7) == [bytes([65 + i]) * 7 for i in range(P)]
c.Barrier()
out = np.zeros(P, np.int64)
rc = _capi.lib().dds_exchange_lenlist(c.handle, 100 + 50 * r, 16, out.ctypes.data_as(_capi.I64P))
assert rc == 0 and out.tolist() == [100, 250], (rc, out)
rc = _capi.lib().dds_exchange_lenlist(c.handle, 5, 16 + r, out.ctypes.data_as(_capi.I64P))
assert (rc == 0) == (r == 1), rc
# the data plane must refuse to exist without a GPU
import torch
if not torch.cuda.is_available():
    try:
        from ddstore_b200 import PyDDStore
        PyDDStore(c)
        raise SystemExit("PyDDStore constructed without a GPU")
    except RuntimeError as e:
        assert "No usable CUDA device" in str(e)
c.Barrier()
dist.destroy_process_group()
print("gloo-ok", r)
"""


def test_torch_distributed_gloo_world2(tmp_path):
    script = tmp_path / "gloo_world2.py"
    script.write_text(GLOO_SCRIPT.format(root=ROOT))
    port = 29500 + (os.getpid() % 2000)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"gloo-ok {r}" in o, o


def test_data_plane_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from ddstore_b200 import PyDDStore
    with pytest.raises(RuntimeError, match="No usable CUDA device"):
        PyDDStore()
    assert _capi.lib().dds_create(None, 0, 0) is None


def test_shm_comm_times_out_instead_of_hanging(monkeypatch):
    """a rank that never arrives must produce an error, not a hang (the reference hangs in MPI_Get / MPI_Win_fence)"""
    import time
    monkeypatch.setenv("DDS_COMM_TIMEOUT_S", "1")
    from ddstore_b200.comm import ShmComm
    key = "to" + uuid.uuid4().hex[:10]
    t0 = time.time()
    with pytest.raises(RuntimeError, match="barrier timed out|timed out"):
        ShmComm(key, 0, 2)  # rank 1 never shows up
    assert time.time() - t0 < 30
    # the creator could not unlink the name (the rendezvous never completed): a later job with the SAME key is told so
    with pytest.raises(RuntimeError, match="stale or mismatched|timed out"):
        ShmComm(key, 0, 2)
    try:
        os.unlink("/dev/shm/dds_b200_" + key)
    except OSError:
        pass


def test_callback_comm_errors_propagate():
    from ddstore_b200.comm import CallbackComm

    def bad_allgather(b):
        raise ValueError("boom")

    c = CallbackComm(0, 2, bad_allgather, lambda: None)
    out = np.zeros(2, np.int64)
    rc = _capi.lib().dds_exchange_lenlist(c.handle, 5, 1, out.ctypes.data_as(_capi.I64P))
    assert rc == _capi.ERR_COMM and "allgather callback failed" in _capi.last_error()
    c.close()


def test_as_dds_comm_accepts_mpi4py_like_objects():
    from ddstore_b200.comm import as_dds_comm

    class FakeMPIComm:  # the four methods of mpi4py.MPI.Comm the adapter uses
        def Get_rank(self):
            return 0

        def Get_size(self):
            return 1

        def allgather(self, b):
            return [b]

        def Barrier(self):
            pass

    c = as_dds_comm(FakeMPIComm())
    assert c.Get_rank() == 0 and c.Get_size() == 1 and c.allgather_bytes(b"xy") == [b"xy"]
    c.Barrier()
    c.close()
    with pytest.raises(TypeError):
        as_dds_comm(object())


def test_public_header_is_plain_c(tmp_path):
    """the drop-in boundary is a C-ABI: include/ddstore_b200.h must compile as C99, not just as C++"""
    src = tmp_path / "use_header.c"
    src.write_text('#include "ddstore_b200.h"\nint main(void) { dds_varinfo_t v; (void)v; return DDS_OK; }\n')
    r = subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"),
                        str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_locate_property_against_oracle_and_reference(coracle):
    """hypothesis: for arbitrary (also degenerate) lenlists and requests, the C-ABI's host lookup and the C oracle agree
    on owner, offset and error class; on seeded random lenlists drawn from the same ranges, both agree with the owner the
    compiled reference returned (tests/golden/reference_cases.json)"""
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=300, deadline=None)
    @given(st.lists(st.integers(0, 40), min_size=1, max_size=12), st.integers(-5, 500), st.integers(0, 60))
    def check(nrows, start, count):
        ll = np.cumsum(np.array(nrows, np.int64))
        t, off, rc = coracle.locate(ll, start, count)
        assert _locate(ll, start, count) == (t, off, rc)
        assert _ss(ll, start) == coracle.sortedsearch(ll, start)

    check()
    for nrows, start, owner in load_reference_cases()["owner_lookup"]:
        ll = np.cumsum(np.array(nrows, np.int64))
        assert _ss(ll, start) == coracle.sortedsearch(ll, start) == owner
