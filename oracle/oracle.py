"""oracle/oracle.py -- TEST INFRASTRUCTURE, not product code.

ctypes loaders for
  * liboracle.so                (oracle/ddstore_oracle.c, the plain-C restatement), class `COracle`
  * _ref/libddstore_ref.so      (the UNMODIFIED reference compiled against oracle/mpi_shim), class `RefWorld`
    (`PortWorld` runs the same timed loops on liboracle.so where _ref is not built)
and an independent NumPy restatement (`np_*` functions) used to cross-check both.

Reference lines followed by the NumPy restatement:
  src/ddstore.cxx:5-17          owner search, incl. the fall-back-to-0
  include/ddstore.hpp:84-89     inclusive scan of the all-gathered row counts
  include/ddstore.hpp:205-214   offset + the two range checks
  include/ddstore.hpp:229-236   byte count and displacement units of the copy
  src/pyddstore.pyx:67-68,86    nrows / disp / count derivation from the ndarray
"""
import ctypes as C
import os
import subprocess
import threading
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_ORACLE = os.path.join(HERE, "liboracle.so")
LIB_REF = os.path.join(HERE, "_ref", "libddstore_ref.so")

ERR_TEXT = {
    1: "Invalid data type",         # include/ddstore.hpp:203
    2: "Invalid start on target",   # include/ddstore.hpp:211
    3: "Invalid count on target",   # include/ddstore.hpp:214
    4: "Invalid disp",              # include/ddstore.hpp:82
}

# dtype codes shared with oracle/ref_driver.cpp (order of the if-chain in src/pyddstore.pyx:69-80)
DTYPES = {np.dtype(np.int32): 0, np.dtype(np.int64): 1, np.dtype(np.uint8): 2,
          np.dtype(np.float32): 3, np.dtype(np.float64): 4, np.dtype(np.bool_): 5}


def build(ref_root="/root/reference"):
    """Compile liboracle.so and, when the reference tree is present, _ref/libddstore_ref.so."""
    subprocess.run(["make", "-s", "-C", HERE, f"REF={ref_root}"], check=True,
                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)


def have_ref():
    return os.path.exists(LIB_REF)


# --------------------------------------------------------------------------- NumPy restatement
def np_sortedsearch(lenlist, num):
    """src/ddstore.cxx:5-17"""
    v = np.asarray(lenlist, dtype=np.int64)
    hit = np.nonzero((v[:-1] <= num) & (num < v[1:]))[0]
    return int(hit[0]) + 1 if hit.size else 0


def np_lenlist(nrows):
    """include/ddstore.hpp:84-89"""
    return np.cumsum(np.asarray(nrows, dtype=np.int64))


def np_locate(lenlist, start, count):
    """include/ddstore.hpp:205-214 -> (target, offset, errcode)"""
    t = np_sortedsearch(lenlist, start)
    off = int(lenlist[t - 1]) if t > 0 else 0
    if start < off:
        return t, off, 2
    if start + count > int(lenlist[t]):
        return t, off, 3
    return t, off, 0


def np_get_batch(shards, starts, counts):
    """shards: list of per-rank 2-D arrays (nrows_r, disp) of one dtype. Returns
    (packed uint8 bytes, int64 offsets[B+1], first_bad, errcode) like the serial get() loop."""
    lenlist = np_lenlist([s.shape[0] for s in shards])
    row = shards[0].dtype.itemsize * (shards[0].size // shards[0].shape[0] if shards[0].shape[0] else
                                      int(np.prod(shards[0].shape[1:], dtype=np.int64)))
    flat = [np.ascontiguousarray(s).view(np.uint8).reshape(-1) for s in shards]
    parts, offs, pos = [], [], 0
    for i, (st, ct) in enumerate(zip(starts, counts)):
        offs.append(pos)
        t, off, err = np_locate(lenlist, int(st), int(ct))
        if err:
            return (np.concatenate(parts) if parts else np.zeros(0, np.uint8)), np.array(offs, np.int64), i, err
        b0 = (int(st) - off) * row
        parts.append(flat[t][b0:b0 + int(ct) * row])
        pos += int(ct) * row
    offs.append(pos)
    out = np.concatenate(parts) if parts else np.zeros(0, np.uint8)
    return out, np.array(offs, np.int64), -1, 0


_MASK = (1 << 64) - 1


def np_synth_rows(seed, first_global_row, nrows, disp, dtype):
    """SURVEY.md 8d payload generator: low itemsize bytes of splitmix64(seed ^ (g*disp + c))."""
    dtype = np.dtype(dtype)
    g = (np.arange(nrows, dtype=np.uint64)[:, None] + np.uint64(first_global_row)) * np.uint64(disp) \
        + np.arange(disp, dtype=np.uint64)[None, :]
    x = (g ^ np.uint64(seed & _MASK)) + np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    x = x ^ (x >> np.uint64(31))
    raw = x.view(np.uint8).reshape(nrows, disp, 8)[:, :, :dtype.itemsize]
    return np.ascontiguousarray(raw).view(dtype).reshape(nrows, disp)


# --------------------------------------------------------------------------- C restatement
class COracle:
    def __init__(self):
        if not os.path.exists(LIB_ORACLE):
            build()
        L = C.CDLL(LIB_ORACLE)
        LP, IP = C.POINTER(C.c_long), C.POINTER(C.c_int)
        L.orc_sortedsearch.argtypes = [LP, C.c_int, C.c_long]
        L.orc_lenlist.argtypes = [LP, IP, C.c_int, LP]
        L.orc_locate.argtypes = [LP, C.c_int, C.c_long, C.c_long, IP, LP]
        L.orc_get.argtypes = [C.POINTER(C.c_void_p), LP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_long, C.c_long,
                              C.c_void_p]
        L.orc_get_batch.argtypes = [C.POINTER(C.c_void_p), LP, C.c_int, C.c_int, C.c_int, C.c_int, LP, LP,
                                    C.c_long, C.c_void_p, LP, LP]
        L.orc_synth_rows.argtypes = [C.c_uint64, C.c_long, C.c_long, C.c_int, C.c_int, C.c_void_p]
        L.orc_synth_rows.restype = None
        self.L = L

    @staticmethod
    def _lp(a):
        return a.ctypes.data_as(C.POINTER(C.c_long))

    def sortedsearch(self, lenlist, num):
        v = np.ascontiguousarray(lenlist, dtype=np.int64)
        return self.L.orc_sortedsearch(self._lp(v), len(v), num)

    def lenlist(self, nrows, disp):
        n = np.ascontiguousarray(nrows, dtype=np.int64)
        d = np.ascontiguousarray(disp, dtype=np.int32)
        out = np.zeros(len(n), np.int64)
        rc = self.L.orc_lenlist(self._lp(n), d.ctypes.data_as(C.POINTER(C.c_int)), len(n), self._lp(out))
        return out, rc

    def locate(self, lenlist, start, count):
        v = np.ascontiguousarray(lenlist, dtype=np.int64)
        t, off = C.c_int(), C.c_long()
        rc = self.L.orc_locate(self._lp(v), len(v), start, count, C.byref(t), C.byref(off))
        return t.value, off.value, rc

    def get_batch(self, shards, starts, counts, req_itemsize=None):
        """Same contract as np_get_batch, run by the C restatement."""
        shards = [np.ascontiguousarray(s) for s in shards]
        itemsize = shards[0].dtype.itemsize
        disp = int(np.prod(shards[0].shape[1:], dtype=np.int64))
        lenlist = np_lenlist([s.shape[0] for s in shards])
        bases = (C.c_void_p * len(shards))(*[s.ctypes.data for s in shards])
        starts = np.ascontiguousarray(starts, dtype=np.int64)
        counts = np.ascontiguousarray(counts, dtype=np.int64)
        cap = int(np.clip(counts, 0, None).sum()) * disp * itemsize
        out = np.zeros(max(cap, 1), np.uint8)
        offs = np.zeros(len(starts) + 1, np.int64)
        bad = C.c_long(-1)
        rc = self.L.orc_get_batch(bases, self._lp(lenlist), len(shards), disp, itemsize,
                                  itemsize if req_itemsize is None else req_itemsize,
                                  self._lp(starts), self._lp(counts), len(starts), out.ctypes.data,
                                  self._lp(offs), C.byref(bad))
        if rc:
            n = int(offs[bad.value])
            return out[:n], offs[:bad.value + 1], bad.value, rc
        return out[:int(offs[-1])], offs, -1, 0

    def synth_rows(self, seed, first_global_row, nrows, disp, dtype):
        dtype = np.dtype(dtype)
        out = np.zeros((nrows, disp), dtype)
        self.L.orc_synth_rows(seed, first_global_row, nrows, disp, dtype.itemsize, out.ctypes.data)
        return out


class PortWorld:
    """`size` thread-ranks of the C restatement with the part of RefWorld's surface a timed get() loop needs (add,
    get_loop_all): the stand-in for the reference where oracle/_ref is not built."""

    def __init__(self, size):
        self.co, self.size, self.vars, self._err = COracle(), size, {}, ""

    def close(self):
        self.vars.clear()

    def err(self):
        return self._err

    def add(self, name, shards):
        shards = [np.ascontiguousarray(s) for s in shards]
        self.vars[name] = (shards, np_lenlist([s.shape[0] for s in shards]))

    def get_loop_all(self, name, starts_per_rank, counts_per_rank, outs):
        """concurrent loops, one thread per rank, each into its packed buffer; returns the wall ns of the slowest
        rank, or -1 with err() set when a request fails"""
        shards, ll = self.vars[name]
        disp = int(np.prod(shards[0].shape[1:], dtype=np.int64))
        itemsize = shards[0].dtype.itemsize
        bases = (C.c_void_p * len(shards))(*[s.ctypes.data for s in shards])
        LP = C.POINTER(C.c_long)
        st = [np.ascontiguousarray(s, dtype=np.int64) for s in starts_per_rank]
        ct = [np.ascontiguousarray(c, dtype=np.int64) for c in counts_per_rank]
        rcs = [0] * self.size

        def one(r):
            rcs[r] = self.co.L.orc_get_batch(bases, ll.ctypes.data_as(LP), len(shards), disp, itemsize, itemsize,
                                             st[r].ctypes.data_as(LP), ct[r].ctypes.data_as(LP), len(st[r]),
                                             outs[r].ctypes.data, None, None)

        th = [threading.Thread(target=one, args=(r,)) for r in range(self.size)]
        t0 = time.perf_counter()
        [t.start() for t in th]
        [t.join() for t in th]
        ns = int((time.perf_counter() - t0) * 1e9)
        bad = [rc for rc in rcs if rc]
        if bad:
            self._err = ERR_TEXT[bad[0]]
            return -1
        return ns


# --------------------------------------------------------------------------- the real reference
class RefWorld:
    """`size` thread-ranks of the unmodified reference DDStore (method 0) over oracle/mpi_shim."""

    def __init__(self, size):
        if not have_ref():
            build()
        if not have_ref():
            raise RuntimeError("oracle/_ref/libddstore_ref.so is not built and /root/reference is absent")
        L = C.CDLL(LIB_REF)
        LP = C.POINTER(C.c_long)
        L.ref_world_create.restype = C.c_void_p
        L.ref_world_create.argtypes = [C.c_int]
        L.ref_world_destroy.argtypes = [C.c_void_p]
        L.ref_last_error.restype = C.c_char_p
        L.ref_last_error.argtypes = [C.c_void_p]
        L.ref_sortedsearch.argtypes = [LP, C.c_int, C.c_long]
        L.ref_add.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.POINTER(C.c_void_p), LP, C.POINTER(C.c_int)]
        L.ref_init.argtypes = [C.c_void_p, C.c_char_p, LP, C.POINTER(C.c_int), C.c_int]
        L.ref_update.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.c_void_p, C.c_long, C.c_long]
        L.ref_get.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.c_long, C.c_long, C.c_void_p]
        L.ref_get_loop.restype = C.c_longlong
        L.ref_get_loop.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int, LP, LP, C.c_long, C.c_long,
                                   C.c_void_p, LP]
        L.ref_get_loop_all.restype = C.c_longlong
        L.ref_get_loop_all.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.POINTER(LP), C.POINTER(LP), C.c_long,
                                       C.c_long, C.POINTER(C.c_void_p)]
        L.ref_epoch_begin.argtypes = [C.c_void_p]
        L.ref_epoch_end.argtypes = [C.c_void_p]
        L.ref_query.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), LP]
        self.L, self.size = L, size
        self.h = L.ref_world_create(size)
        self.vars = {}

    def close(self):
        if self.h:
            self.L.ref_world_destroy(self.h)
            self.h = None

    def err(self):
        return self.L.ref_last_error(self.h).decode()

    def sortedsearch(self, lenlist, num):
        v = np.ascontiguousarray(lenlist, dtype=np.int64)
        return self.L.ref_sortedsearch(v.ctypes.data_as(C.POINTER(C.c_long)), len(v), num)

    def add(self, name, shards):
        """collective add on all ranks; shards[r] is rank r's 2-D array (src/pyddstore.pyx:65-82)."""
        shards = [np.ascontiguousarray(s) for s in shards]
        nrows = np.array([s.shape[0] for s in shards], np.int64)
        disp = np.array([(s.size // s.shape[0]) if s.shape[0] else int(np.prod(s.shape[1:], dtype=np.int64))
                         for s in shards], np.int32)
        bufs = (C.c_void_p * self.size)(*[s.ctypes.data for s in shards])
        rc = self.L.ref_add(self.h, name.encode(), DTYPES[shards[0].dtype], bufs,
                            nrows.ctypes.data_as(C.POINTER(C.c_long)), disp.ctypes.data_as(C.POINTER(C.c_int)))
        if rc:
            raise ValueError(self.err())
        self.vars[name] = (shards[0].dtype, int(disp[0]))

    def init(self, name, nrows, disp, itemsize, dtype):
        n = np.ascontiguousarray(nrows, dtype=np.int64)
        d = np.ascontiguousarray(disp, dtype=np.int32)
        rc = self.L.ref_init(self.h, name.encode(), n.ctypes.data_as(C.POINTER(C.c_long)),
                             d.ctypes.data_as(C.POINTER(C.c_int)), itemsize)
        if rc:
            raise ValueError(self.err())
        self.vars[name] = (np.dtype(dtype), int(d[0]))

    def update(self, rank, name, arr, offset):
        arr = np.ascontiguousarray(arr)
        rc = self.L.ref_update(self.h, rank, name.encode(), DTYPES[arr.dtype], arr.ctypes.data, arr.shape[0], offset)
        if rc:
            raise ValueError(self.err())

    def get(self, rank, name, arr, start):
        """src/pyddstore.pyx:84-101: count = arr.shape[0]; fills arr in place."""
        rc = self.L.ref_get(self.h, rank, name.encode(), DTYPES[arr.dtype], start, arr.shape[0], arr.ctypes.data)
        if rc:
            raise ValueError(self.err())

    def get_batch(self, rank, name, starts, counts):
        """serial get() loop; returns (packed uint8, first_bad, error text or None, elapsed ns)."""
        dtype, disp = self.vars[name]
        row = disp * dtype.itemsize
        starts = np.ascontiguousarray(starts, dtype=np.int64)
        counts = np.ascontiguousarray(counts, dtype=np.int64)
        out = np.zeros(max(int(np.clip(counts, 0, None).sum()) * row, 1), np.uint8)
        bad = C.c_long(-1)
        LP = C.POINTER(C.c_long)
        ns = self.L.ref_get_loop(self.h, rank, name.encode(), DTYPES[dtype], starts.ctypes.data_as(LP),
                                 counts.ctypes.data_as(LP), len(starts), row, out.ctypes.data, C.byref(bad))
        if ns < 0:
            n = int(counts[:bad.value].sum()) * row
            return out[:n], bad.value, self.err(), ns
        return out[:int(counts.sum()) * row], -1, None, ns

    def get_loop_all(self, name, starts_per_rank, counts_per_rank, outs):
        """timed concurrent loops, one thread per rank; returns slowest rank's ns."""
        dtype, disp = self.vars[name]
        row = disp * dtype.itemsize
        LP = C.POINTER(C.c_long)
        st = [np.ascontiguousarray(s, dtype=np.int64) for s in starts_per_rank]
        ct = [np.ascontiguousarray(c, dtype=np.int64) for c in counts_per_rank]
        sp = (LP * self.size)(*[s.ctypes.data_as(LP) for s in st])
        cp = (LP * self.size)(*[c.ctypes.data_as(LP) for c in ct])
        op = (C.c_void_p * self.size)(*[o.ctypes.data for o in outs])
        return self.L.ref_get_loop_all(self.h, name.encode(), DTYPES[dtype], sp, cp, len(st[0]), row, op)

    def epoch_begin(self):
        if self.L.ref_epoch_begin(self.h):
            raise RuntimeError(self.err())

    def epoch_end(self):
        if self.L.ref_epoch_end(self.h):
            raise RuntimeError(self.err())

    def query(self, rank, name):
        it, dp = C.c_int(), C.c_int()
        ll = np.zeros(self.size, np.int64)
        rc = self.L.ref_query(self.h, rank, name.encode(), C.byref(it), C.byref(dp),
                              ll.ctypes.data_as(C.POINTER(C.c_long)))
        if rc:
            raise KeyError(name)
        return it.value, dp.value, ll
