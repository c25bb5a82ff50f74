"""Host-side mirror of DBoW2's ORBVocabulary::transform (reference code/Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:
1151-1218) on top of the C ABI: Frame::ComputeBoW / KeyFrame::ComputeBoW (code/src/Frame.cc:445-452,
code/src/KeyFrame.cc:126-133) for one frame, a batch of frames, or a device-resident frame."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import BowOut, SwmError, ptr

__all__ = ["ORBVocabulary", "BowResult", "bow_csr"]


class BowResult:
    """BowVector (word_ids ascending, values) and FeatureVector (CSR: node_ids ascending, offsets, feats) of a frame."""

    def __init__(self, word_ids, values, node_ids, offsets, feats):
        self.word_ids, self.values = word_ids, values
        self.node_ids, self.offsets, self.feats = node_ids, offsets, feats

    def feature_vector(self):
        """The FeatureVector in the form ORBmatcher.SearchByBoW takes."""
        from .matcher import FeatureVector
        fv = FeatureVector.__new__(FeatureVector)
        fv.node_ids = np.ascontiguousarray(self.node_ids, np.uint32)
        fv.offsets = np.ascontiguousarray(self.offsets, np.int32)
        fv.feats = np.ascontiguousarray(self.feats, np.uint32)
        return fv


def bow_csr(bows):
    """A list of BowVectors (BowResult objects or (word_ids, values) pairs) -> (offsets int32, words uint32,
    values float64)."""
    pairs = [(b.word_ids, b.values) if hasattr(b, "word_ids") else b for b in bows]
    off = np.zeros(len(pairs) + 1, np.int32)
    off[1:] = np.cumsum([len(w) for w, _ in pairs])
    words = np.ascontiguousarray(np.concatenate([np.asarray(w, np.uint32) for w, _ in pairs]) if pairs else
                                 np.zeros(0, np.uint32), np.uint32)
    values = np.ascontiguousarray(np.concatenate([np.asarray(v, np.float64) for _, v in pairs]) if pairs else
                                  np.zeros(0, np.float64), np.float64)
    return off, words, values


class ORBVocabulary:
    def __init__(self, blob, device=0):
        """blob: bytes of a vocabulary in the ORBvoc.bin layout (TemplatedVocabulary.h:1478-1522)."""
        self._lib = _lib.load()
        self._blob = np.frombuffer(blob, np.uint8)
        self._h = C.c_void_p()
        rc = self._lib.swm_vocab_create(int(device), ptr(self._blob), len(self._blob), C.byref(self._h))
        if rc != 0:
            msg = self._lib.swm_vocab_last_error(None)
            raise SwmError(f"swm_vocab_create: {_lib.ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")
        a = [C.c_int32() for _ in range(4)]
        self._lib.swm_vocab_info(self._h, *[C.byref(x) for x in a])
        self.k, self.L, self.n_nodes, self.n_words = [x.value for x in a]

    def close(self):
        if getattr(self, "_h", None):
            self._lib.swm_vocab_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            msg = self._lib.swm_vocab_last_error(self._h)
            raise SwmError(f"{what}: {_lib.ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")

    @staticmethod
    def _alloc(batch, cap):
        o = dict(word_ids=np.zeros((batch, cap), np.uint32), word_values=np.zeros((batch, cap), np.float64),
                 n_words=np.zeros(batch, np.int32), node_ids=np.zeros((batch, cap), np.uint32),
                 node_offsets=np.zeros((batch, cap + 1), np.int32), feats=np.zeros((batch, cap), np.uint32),
                 n_nodes=np.zeros(batch, np.int32))
        view = BowOut(*[ptr(o[k]).value for k in ("word_ids", "word_values", "n_words", "node_ids", "node_offsets",
                                                   "feats", "n_nodes")])
        return o, view

    @staticmethod
    def _result(o, b):
        nw, nn = int(o["n_words"][b]), int(o["n_nodes"][b])
        off = o["node_offsets"][b, :nn + 1].copy()
        return BowResult(o["word_ids"][b, :nw].copy(), o["word_values"][b, :nw].copy(), o["node_ids"][b, :nn].copy(), off,
                         o["feats"][b, :off[nn] if nn else 0].copy())

    def transform_batch(self, desc, n, levelsup=4):
        """desc: (B, cap, 32) uint8 host array, n: (B,) valid rows.  Returns a list of BowResult."""
        desc = np.ascontiguousarray(desc, np.uint8)
        n = np.ascontiguousarray(n, np.int32)
        batch, cap = desc.shape[0], desc.shape[1]
        o, view = self._alloc(batch, cap)
        self._check(self._lib.swm_bow_transform(self._h, ptr(desc), ptr(n), batch, cap, int(levelsup), C.byref(view)),
                    "swm_bow_transform")
        return [self._result(o, b) for b in range(batch)]

    def transform(self, desc, levelsup=4):
        """mpORBvocabulary->transform(vCurrentDesc, mBowVec, mFeatVec, 4) for one frame's (N, 32) descriptors."""
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        if len(desc) == 0:
            z = np.zeros(0, np.uint32)
            return BowResult(z, np.zeros(0), z, np.zeros(1, np.int32), z)
        return self.transform_batch(desc[None], np.array([len(desc)], np.int32), levelsup)[0]

    def score_pairs(self, a, b):
        """ORBVocabulary::score (DBoW2 L1Scoring::score) of each pair (a[i], b[i]) of BowVectors: BowResult objects or
        (word_ids, values) pairs.  L1_NORM vocabularies only.  Returns float64 scores, bit-exact."""
        if len(a) != len(b):
            raise ValueError("a and b must hold the same number of BowVectors")
        ao, aw, av = bow_csr(a)
        bo, bw, bv = bow_csr(b)
        out = np.zeros(len(a), np.float64)
        self._check(self._lib.swm_bow_score(self._h, len(a), ptr(ao), ptr(aw), ptr(av), ptr(bo), ptr(bw), ptr(bv),
                                            ptr(out)), "swm_bow_score")
        return out

    def score(self, a, b):
        """ORBVocabulary::score(a, b) of two BowVectors."""
        return float(self.score_pairs([a], [b])[0])

    def transform_frame(self, frame, levelsup=4):
        """The same for a ResidentFrame: the descriptors stay on the device."""
        cap = max(frame.N, 1)
        o, view = self._alloc(1, cap)
        self._check(self._lib.swm_bow_transform_frame(self._h, frame._h, int(levelsup), C.byref(view)),
                    "swm_bow_transform_frame")
        return self._result(o, 0)
