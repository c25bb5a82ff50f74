"""ctypes binding of the KeyFrameDatabase oracle (oracle/liborb_oracle_kfdb.so, oracle/orb_oracle_kfdb.cpp).

TEST INFRASTRUCTURE: imported by tests/, __graft_entry__ and tools/kfdb_probe.py only; the product package never
imports it."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(_HERE), "oracle")
SO = os.path.join(ORACLE_DIR, "liborb_oracle_kfdb.so")
SRCS = [os.path.join(ORACLE_DIR, f) for f in ("orb_oracle_kfdb.cpp", "orb_oracle_kfdb.h")]
# the flags of oracle/Makefile: no FMA contraction, so the float / double sums round as the reference's do
CXX_FLAGS = ["-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-Wall", "-Wextra", "-shared"]

_lib = None
_p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731


def build(force=False):
    if force or not os.path.exists(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in SRCS):
        subprocess.run([os.environ.get("CXX", "g++")] + CXX_FLAGS + ["-o", SO, SRCS[0]], check=True,
                       capture_output=True)
    return SO


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        vp, ci, cf, u64 = C.c_void_p, C.c_int, C.c_float, C.c_uint64
        L.orc_l1_score.argtypes = [ci, vp, vp, ci, vp, vp]
        L.orc_l1_score.restype = C.c_double
        L.orc_kfdb_create.argtypes = [ci]
        L.orc_kfdb_create.restype = vp
        L.orc_kfdb_destroy.argtypes = [vp]
        L.orc_kfdb_add.argtypes = [vp, u64, ci, vp, vp]
        L.orc_kfdb_erase.argtypes = [vp, u64]
        L.orc_kfdb_clear.argtypes = [vp]
        L.orc_kfdb_size.argtypes = [vp]
        L.orc_kfdb_set_neighbours.argtypes = [vp, ci, vp, vp, vp]
        L.orc_kfdb_query.argtypes = [vp, ci, ci, vp, vp, cf, ci, vp, vp, vp, ci, vp, vp, ci]
        L.orc_kfdb_time_queries.argtypes = [vp, ci, ci, vp, vp, vp, vp, ci]
        L.orc_kfdb_time_queries.restype = C.c_double
        _lib = L
    return _lib


def _bow(b):
    """(word_ids, values) or any object with .word_ids / .values (a BowResult)."""
    w, v = (b.word_ids, b.values) if hasattr(b, "word_ids") else b
    return np.ascontiguousarray(w, np.uint32), np.ascontiguousarray(v, np.float64)


def l1_score(a, b):
    aw, av = _bow(a)
    bw, bv = _bow(b)
    return lib().orc_l1_score(len(aw), _p(aw), _p(av), len(bw), _p(bw), _p(bv))


class KeyFrameDatabase:
    """The oracle database.  neighbours: {id: ordered best-10 ids}, the GetBestCovisibilityKeyFrames(10) table."""

    def __init__(self, n_words):
        self._h = lib().orc_kfdb_create(int(n_words))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_kfdb_destroy(self._h)
            self._h = None

    def add(self, kf_id, bow):
        w, v = _bow(bow)
        return lib().orc_kfdb_add(self._h, int(kf_id), len(w), _p(w), _p(v))

    def erase(self, kf_id):
        lib().orc_kfdb_erase(self._h, int(kf_id))

    def clear(self):
        lib().orc_kfdb_clear(self._h)

    def size(self):
        return lib().orc_kfdb_size(self._h)

    def set_neighbours(self, neighbours):
        ids = np.array(list(neighbours.keys()), np.uint64)
        lens = [len(neighbours[int(i)]) for i in ids]
        off = np.zeros(len(ids) + 1, np.int32)
        off[1:] = np.cumsum(lens)
        nb = np.array([x for i in ids for x in neighbours[int(i)]], np.uint64)
        lib().orc_kfdb_set_neighbours(self._h, len(ids), _p(ids), _p(off), _p(nb))

    def query(self, mode, bow, min_score=0.0, connected=()):
        """-> (scored ids, scored float32 scores, candidate ids): lScoreAndMatch in list order and the result."""
        w, v = _bow(bow)
        conn = np.array(list(connected), np.uint64)
        cap = self.size() + 1
        sid, ssc, cid = np.zeros(cap, np.uint64), np.zeros(cap, np.float32), np.zeros(cap, np.uint64)
        ns = C.c_int(0)
        nc = lib().orc_kfdb_query(self._h, int(mode), len(w), _p(w), _p(v), float(min_score), len(conn), _p(conn),
                                  _p(sid), _p(ssc), cap, C.byref(ns), _p(cid), cap)
        return sid[:ns.value], ssc[:ns.value], cid[:nc]

    def reloc(self, bow):
        return self.query(0, bow)

    def loop(self, bow, min_score, connected=()):
        return self.query(1, bow, min_score, connected)

    def time_queries(self, mode, bows, min_scores, iters):
        off = np.zeros(len(bows) + 1, np.int32)
        off[1:] = np.cumsum([len(_bow(b)[0]) for b in bows])
        w = np.concatenate([_bow(b)[0] for b in bows]) if bows else np.zeros(0, np.uint32)
        v = np.concatenate([_bow(b)[1] for b in bows]) if bows else np.zeros(0, np.float64)
        ms = np.ascontiguousarray(min_scores, np.float32)
        return lib().orc_kfdb_time_queries(self._h, int(mode), len(bows), _p(off), _p(w), _p(v), _p(ms), int(iters))
