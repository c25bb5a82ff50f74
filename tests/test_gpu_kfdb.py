"""KeyFrameDatabase on the GPU (swarmmap_b200.kfdb, csrc/kfdb.cu) against the CPU oracle (oracle/orb_oracle_kfdb.cpp):
ordered scored lists with bit-equal float scores, ordered candidate lists, batched queries equal to the same queries
issued one by one, stale reloc scores within a batch and across calls, add / erase / re-add between queries, a 10 k
keyframe database, ORBVocabulary.score bit-exact, and the error paths."""
import numpy as np
import pytest

import oracle_kfdb_lib as okl
from swarmmap_b200 import synth

pytestmark = pytest.mark.gpu


def random_bow(rng, n_words, n):
    w = np.sort(rng.choice(n_words, n, replace=False)).astype(np.uint32)
    v = rng.random(n)
    return w, v / v.sum()


def bow(words, values=None):
    w = np.array(sorted(words), np.uint32)
    v = np.full(len(w), 1.0 / max(len(w), 1)) if values is None else np.asarray(values, np.float64)
    return w, v


@pytest.fixture(scope="module")
def vocab(swm):
    from swarmmap_b200.bow import ORBVocabulary
    return ORBVocabulary(synth.make_vocabulary(10, 3, seed=11))  # L1_NORM, ~1000 words


class Pair:
    """The device database and the oracle fed the same operations."""

    def __init__(self, vocab, neighbours):
        from swarmmap_b200.kfdb import KeyFrameDatabase
        self.g, self.o, self.nb = KeyFrameDatabase(vocab), okl.KeyFrameDatabase(vocab.n_words), neighbours
        self.o.set_neighbours(neighbours)

    def add(self, ids, bows):
        self.g.add(ids, bows)
        for i, b in zip(ids, bows):
            assert self.o.add(i, b) == 0

    def erase(self, ids):
        self.g.erase(ids)
        for i in ids:
            self.o.erase(i)

    def clear(self):
        self.g.clear()
        self.o.clear()

    def check(self, mode, queries, min_scores=None, connected=None):
        """One device batch against the oracle's queries issued in order; returns the candidate lists."""
        if mode == 0:
            cand = self.g.detect_relocalization_candidates(queries, self.nb)
        else:
            cand = self.g.detect_loop_candidates(queries, min_scores, connected, self.nb)
        for q, b in enumerate(queries):
            sid, ssc, cid = self.o.query(mode, b, 0.0 if mode == 0 else min_scores[q], () if mode == 0 else connected[q])
            gid, gsc = self.g.last_scored[q]
            np.testing.assert_array_equal(gid, sid)
            np.testing.assert_array_equal(gsc.view(np.uint32), ssc.view(np.uint32))  # float bits
            np.testing.assert_array_equal(cand[q], cid)
        return cand


def make_db(rng, n_kf, n_words, words_per_kf):
    ids = rng.choice(10 ** 9, n_kf, replace=False).astype(np.uint64)
    bows = [random_bow(rng, n_words, int(rng.integers(words_per_kf // 2, words_per_kf))) for _ in range(n_kf)]
    nb = {int(i): [int(x) for x in rng.choice(ids, int(rng.integers(0, 11)), replace=False)] for i in ids}
    return ids, bows, nb


def queries_for(rng, bows, n_words, n, words):
    """Re-renders of database keyframes (a few words swapped) and fresh random vectors."""
    out = []
    for _ in range(n):
        if rng.random() < 0.6:
            w, v = bows[int(rng.integers(len(bows)))]
            keep = rng.random(len(w)) < 0.8
            extra = rng.choice(n_words, 5, replace=False)
            ww = np.unique(np.concatenate([w[keep], extra])).astype(np.uint32)
            out.append((ww, rng.random(len(ww)) / len(ww)))
        else:
            out.append(random_bow(rng, n_words, words))
    return out


def test_bow_score_bit_exact(vocab):
    rng = np.random.default_rng(1)
    a = [random_bow(rng, vocab.n_words, int(rng.integers(0, 300))) for _ in range(300)]
    b = [random_bow(rng, vocab.n_words, int(rng.integers(0, 300))) for _ in range(300)]
    got = vocab.score_pairs(a, b)
    ref = np.array([okl.l1_score(x, y) for x, y in zip(a, b)])
    np.testing.assert_array_equal(got.view(np.uint64), ref.view(np.uint64))
    assert vocab.score(a[0], a[0]) == okl.l1_score(a[0], a[0])


def test_reloc_batches_with_stale_scores(vocab):
    """Consecutive reloc batches over one database: sharing-but-unscored neighbours read scores from earlier queries
    of the same batch and from earlier calls."""
    rng = np.random.default_rng(2)
    ids, bows, nb = make_db(rng, 400, vocab.n_words, 60)
    d = Pair(vocab, nb)
    d.add(ids, bows)
    n_cand = 0
    for step in range(6):
        qs = queries_for(rng, bows, vocab.n_words, [1, 16, 64, 5, 128, 33][step], 50)
        n_cand += sum(len(c) for c in d.check(0, qs))
    assert n_cand > 0


def test_hand_built_stale_score_in_batch_and_across_calls(vocab):
    from swarmmap_b200.kfdb import KeyFrameDatabase
    nb = {1: [9]}
    q2, q9 = bow([1, 2, 3, 4, 5, 6, 7, 8]), bow([1, 20, 21, 22])
    g = KeyFrameDatabase(vocab)
    g.add([1, 9], [bow([1, 2, 3, 4, 5, 6, 7, 8], [0.05] * 8), bow([1, 20, 21, 22])])
    # within one batch: initial 0.0f, then keyframe 9 is scored by the second query and stale in the third
    c = g.detect_relocalization_candidates([q2, q9, q2], nb)
    assert [x.tolist() for x in c] == [[1], [9], [9]]
    # across calls on a fresh database: the same
    g2 = KeyFrameDatabase(vocab)
    g2.add([1, 9], [bow([1, 2, 3, 4, 5, 6, 7, 8], [0.05] * 8), bow([1, 20, 21, 22])])
    assert [g2.detect_relocalization_candidates([q], nb)[0].tolist() for q in (q2, q9, q2)] == [[1], [9], [9]]
    # the state survives erase, re-add and clear
    g2.erase([9])
    g2.clear()
    g2.add([1, 9], [bow([1, 2, 3, 4, 5, 6, 7, 8], [0.05] * 8), bow([1, 20, 21, 22])])
    assert g2.detect_relocalization_candidates([q2], nb)[0].tolist() == [9]


def test_batch_equals_single_calls(vocab):
    from swarmmap_b200.kfdb import KeyFrameDatabase
    rng = np.random.default_rng(3)
    ids, bows, nb = make_db(rng, 300, vocab.n_words, 50)
    qs = queries_for(rng, bows, vocab.n_words, 40, 40)
    ms = rng.random(40).astype(np.float32) * 0.05
    conn = [rng.choice(ids, 5, replace=False).tolist() for _ in range(40)]
    a, b = KeyFrameDatabase(vocab), KeyFrameDatabase(vocab)
    a.add(ids, bows)
    b.add(ids, bows)
    for mode in (0, 1):
        if mode == 0:
            batch = a.detect_relocalization_candidates(qs, nb)
            single = [b.detect_relocalization_candidates([q], nb)[0] for q in qs]
        else:
            batch = a.detect_loop_candidates(qs, ms, conn, nb)
            single = [b.detect_loop_candidates([q], ms[i:i + 1], [conn[i]], nb)[0] for i, q in enumerate(qs)]
        for x, y in zip(batch, single):
            np.testing.assert_array_equal(x, y)


def test_loop_and_reloc_with_add_erase_readd(vocab):
    rng = np.random.default_rng(4)
    ids, bows, nb = make_db(rng, 300, vocab.n_words, 60)
    idl = [int(i) for i in ids]
    d = Pair(vocab, nb)
    d.add(ids[:200], bows[:200])
    for step in range(8):
        qs = queries_for(rng, bows, vocab.n_words, 24, 40)
        if step % 2:
            ms = (rng.random(len(qs)) * 0.05).astype(np.float32)
            conn = [rng.choice(ids, int(rng.integers(0, 12)), replace=False).tolist() for _ in qs]
            d.check(1, qs, ms, conn)
        else:
            d.check(0, qs)
        if step == 2:
            gone = rng.choice(200, 20, replace=False)
            d.erase([idl[k] for k in gone])
            d.add([idl[k] for k in gone[:10]], [bows[k] for k in gone[:10]])  # re-added: back of every list
        if step == 5:
            d.clear()
            d.add(ids[100:], bows[100:])
        if step == 6:
            d.erase([12345, int(ids[150])])  # an unknown id is a no-op
    assert len(d.g) == d.o.size()


def test_ten_thousand_keyframes_sampled_queries(swm):
    from swarmmap_b200.bow import ORBVocabulary
    vocab = ORBVocabulary(synth.make_vocabulary(10, 4, seed=12))  # ~10 k words
    rng = np.random.default_rng(5)
    ids, bows, nb = make_db(rng, 10000, vocab.n_words, 300)
    d = Pair(vocab, nb)
    d.add(ids, bows)
    qs = queries_for(rng, bows, vocab.n_words, 48, 250)
    d.check(0, qs)
    d.check(1, qs, np.full(len(qs), 0.01, np.float32), [rng.choice(ids, 10).tolist() for _ in qs])


def test_errors(swm, vocab):
    from swarmmap_b200._lib import SwmError
    from swarmmap_b200.bow import ORBVocabulary
    from swarmmap_b200.kfdb import KeyFrameDatabase
    l2 = ORBVocabulary(synth.make_vocabulary(10, 2, seed=1, scoring=1))
    with pytest.raises(SwmError, match="L1_NORM"):
        KeyFrameDatabase(l2)
    with pytest.raises(SwmError, match="L1_NORM"):
        l2.score(bow([1]), bow([1]))
    g = KeyFrameDatabase(vocab)
    g.add([7], [bow([1, 2])])
    with pytest.raises(SwmError, match="SWM_E_INVALID"):
        g.add([7], [bow([3])])                       # duplicate live id
    with pytest.raises(SwmError, match="SWM_E_INVALID"):
        g.add([8, 8], [bow([3]), bow([4])])          # duplicate inside one call
    with pytest.raises(SwmError, match="SWM_E_INVALID"):
        g.add([9], [bow([vocab.n_words])])           # word id out of range
    assert len(g) == 1
    with pytest.raises(SwmError, match="SWM_E_STATE"):
        g.finish({})                                 # finish before any query
    g.last_scored = None
    g.query(0, [bow([1, 2])])
    g.add([10], [bow([1, 2])])
    with pytest.raises(SwmError, match="SWM_E_STATE"):
        g.finish({})                                 # add between query and finish
    # capacity: the C entry points report the size needed and change nothing
    from swarmmap_b200._lib import ptr
    q_off, qw, qv = np.array([0, 2], np.int32), np.array([1, 2], np.uint32), np.array([0.5, 0.5])
    so, sid, ssc = np.zeros(2, np.int32), np.zeros(1, np.uint64), np.zeros(1, np.float32)
    lib = swm.load()
    rc = lib.swm_kfdb_query(g._h, 0, 1, ptr(q_off), ptr(qw), ptr(qv), None, None, None, ptr(so), ptr(sid), ptr(ssc), 1)
    assert rc == -4 and so[1] == 2
    rc = lib.swm_kfdb_finish(g._h, ptr(np.zeros(3, np.int32)), None, ptr(np.zeros(2, np.int32)), None, 0)
    assert rc == -5                                  # the failed query left nothing to finish
    sid, ssc = np.zeros(2, np.uint64), np.zeros(2, np.float32)
    assert lib.swm_kfdb_query(g._h, 0, 1, ptr(q_off), ptr(qw), ptr(qv), None, None, None, ptr(so), ptr(sid), ptr(ssc),
                              2) == 0
    co, cid = np.zeros(2, np.int32), np.zeros(2, np.uint64)
    rc = lib.swm_kfdb_finish(g._h, ptr(np.zeros(3, np.int32)), None, ptr(co), ptr(cid), 0)
    assert rc == -4 and co[1] == 2
    assert lib.swm_kfdb_finish(g._h, ptr(np.zeros(3, np.int32)), None, ptr(co), ptr(cid), 2) == 0
    assert sorted(cid.tolist()) == [7, 10]
