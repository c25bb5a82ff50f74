"""Host-side mirror of ORB-SLAM2's KeyFrameDatabase (as SwarmMap carries it) on top of the C ABI (swm_kfdb_*):
DetectRelocalizationCandidates (Tracking::Relocalization) and DetectLoopCandidates (LoopClosing::DetectLoop,
AgentMediator::CheckOverlapCandidates) with DBoW2's L1 score, on the GPU.  A batch of queries equals the same queries
issued one after another; the rules and frozen definitions are in DESIGN.md section 2."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import SwmError, ptr
from .bow import bow_csr

__all__ = ["KeyFrameDatabase", "RELOC", "LOOP"]

RELOC, LOOP = 0, 1


def _neighbour_fn(neighbours):
    if callable(neighbours):
        return neighbours
    return lambda i: neighbours.get(i, ())


class KeyFrameDatabase:
    def __init__(self, vocab):
        """vocab: a swarmmap_b200.bow.ORBVocabulary with L1_NORM scoring (ORBvoc's)."""
        self._lib = _lib.load()
        self._vocab = vocab  # the database uses the vocabulary's device; keep it alive
        self._h = C.c_void_p()
        rc = self._lib.swm_kfdb_create(vocab._h, C.byref(self._h))
        if rc != 0:
            msg = self._lib.swm_kfdb_last_error(None)
            raise SwmError(f"swm_kfdb_create: {_lib.ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")
        self.last_scored = None

    def close(self):
        if getattr(self, "_h", None):
            self._lib.swm_kfdb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            msg = self._lib.swm_kfdb_last_error(self._h)
            raise SwmError(f"{what}: {_lib.ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")

    def __len__(self):
        return int(self._lib.swm_kfdb_size(self._h))

    def add(self, ids, bows):
        """KeyFrameDatabase::add for each keyframe: ids[i] with BowVector bows[i] (BowResult or (word_ids, values))."""
        ids = np.ascontiguousarray(ids, np.uint64).reshape(-1)
        off, w, v = bow_csr(bows)
        if len(ids) != len(off) - 1:
            raise ValueError("one BowVector per id")
        self._check(self._lib.swm_kfdb_add(self._h, len(ids), ptr(ids), ptr(off), ptr(w), ptr(v)), "swm_kfdb_add")

    def erase(self, ids):
        ids = np.ascontiguousarray(ids, np.uint64).reshape(-1)
        self._check(self._lib.swm_kfdb_erase(self._h, len(ids), ptr(ids)), "swm_kfdb_erase")

    def clear(self):
        self._check(self._lib.swm_kfdb_clear(self._h), "swm_kfdb_clear")

    def query(self, mode, queries, min_scores=None, connected=None):
        """Phase 1: -> list per query of (scored ids uint64, float32 scores), lScoreAndMatch in list order."""
        nq = len(queries)
        off, w, v = bow_csr(queries)
        ms = np.zeros(nq, np.float32) if min_scores is None else np.ascontiguousarray(min_scores, np.float32)
        coff, cids = None, np.zeros(1, np.uint64)
        if connected is not None:
            conn = [np.asarray(list(c), np.uint64) for c in connected]
            coff = np.zeros(nq + 1, np.int32)
            coff[1:] = np.cumsum([len(c) for c in conn])
            cids = np.ascontiguousarray(np.concatenate(conn) if conn else np.zeros(0, np.uint64), np.uint64)
        so = np.zeros(nq + 1, np.int32)
        cap = max(len(self), 1)
        while True:
            sid, ssc = np.zeros(cap, np.uint64), np.zeros(cap, np.float32)
            rc = self._lib.swm_kfdb_query(self._h, int(mode), nq, ptr(off), ptr(w), ptr(v), ptr(ms),
                                          ptr(coff) if coff is not None else None, ptr(cids), ptr(so), ptr(sid),
                                          ptr(ssc), cap)
            if rc == -4 and int(so[nq]) > cap:  # SWM_E_CAPACITY: nothing changed, repeat with the size needed
                cap = int(so[nq])
                continue
            self._check(rc, "swm_kfdb_query")
            break
        self.last_scored = [(sid[so[q]:so[q + 1]].copy(), ssc[so[q]:so[q + 1]].copy()) for q in range(nq)]
        return self.last_scored

    def finish(self, neighbours):
        """Phase 2: neighbours (mapping or callable id -> ordered GetBestCovisibilityKeyFrames(10) ids) of the scored
        entries of the last query -> list per query of candidate ids (uint64)."""
        fn = _neighbour_fn(neighbours)
        scored = self.last_scored or []
        flat = [np.asarray(list(fn(int(i))), np.uint64) for sid, _ in scored for i in sid]
        noff = np.zeros(len(flat) + 1, np.int32)
        noff[1:] = np.cumsum([len(x) for x in flat])
        nids = np.ascontiguousarray(np.concatenate(flat) if flat else np.zeros(0, np.uint64), np.uint64)
        nq = max(len(scored), 1)
        co = np.zeros(nq + 1, np.int32)
        cap = max(int(noff.size - 1), 1)
        cid = np.zeros(cap, np.uint64)
        self._check(self._lib.swm_kfdb_finish(self._h, ptr(noff), ptr(nids), ptr(co), ptr(cid), cap), "swm_kfdb_finish")
        return [cid[co[q]:co[q + 1]].copy() for q in range(nq)]

    def detect_relocalization_candidates(self, queries, neighbours):
        """DetectRelocalizationCandidates for each query BowVector, issued in order: list of candidate id arrays."""
        self.query(RELOC, queries)
        return self.finish(neighbours)

    def detect_loop_candidates(self, queries, min_scores, connected, neighbours):
        """DetectLoopCandidates(pKF, minScore) for each query: connected[q] = GetConnectedKeyFrames() ids of query q."""
        self.query(LOOP, queries, min_scores, connected)
        return self.finish(neighbours)

    def last_device_ms(self):
        return float(self._lib.swm_kfdb_last_device_ms(self._h))
