"""Second reading of KeyFrameDatabase (oracle/orb_oracle_kfdb.cpp): a pure-Python restatement written from the rules
in DESIGN.md section 2, not from the C++.  It keeps no inverted lists: the list order of a query is the sort of
(position of the first common word in the query, add sequence number), and the word count is the size of the word
intersection.  Compared with the oracle on random databases, plus one hand-built case per rule whose expected
result changes when that rule changes."""
import numpy as np
import pytest

import oracle_kfdb_lib as okl

F32 = np.float32


def l1(a, b):
    aw, av = a
    bd = dict(zip(b[0].tolist(), b[1].tolist()))
    s = 0.0
    for w, x in zip(aw.tolist(), av.tolist()):
        if w in bd:
            y = bd[w]
            s += abs(x - y) - abs(x) - abs(y)
    return -s / 2.0


class Model:
    def __init__(self, n_words):
        self.n_words, self.live, self.seq, self.reloc_score = n_words, {}, 0, {}

    def add(self, i, bow):
        w = np.asarray(bow[0])
        if i in self.live or (len(w) and (w.max() >= self.n_words or np.any(np.diff(w.astype(np.int64)) <= 0))):
            return -1
        self.seq += 1
        self.live[i] = (self.seq, (np.asarray(bow[0], np.uint32), np.asarray(bow[1], np.float64)))
        return 0

    def erase(self, i):
        self.live.pop(i, None)

    def clear(self):
        self.live.clear()

    def query(self, mode, bow, min_score=0.0, connected=(), neighbours=None):
        neighbours = neighbours or {}
        qpos = {int(w): p for p, w in enumerate(bow[0].tolist())}
        share = {}
        for i, (seq, b) in self.live.items():
            common = sorted(set(b[0].tolist()) & set(qpos))
            if common and not (mode == 1 and i in connected):
                share[i] = (qpos[common[0]], seq, len(common))
        order = sorted(share, key=lambda i: share[i][:2])
        if not order:
            return [], [], []
        min_common = int(F32(max(v[2] for v in share.values())) * F32(0.8))
        scored, entries = {}, []
        for i in order:
            if share[i][2] > min_common:
                s = F32(l1(bow, self.live[i][1]))
                scored[i] = s
                if mode == 0:
                    self.reloc_score[i] = s
                if mode == 0 or s >= F32(min_score):
                    entries.append((i, s))
        acc_best, best_acc = [], F32(0.0) if mode == 0 else F32(min_score)
        for i, s in entries:
            acc, best, best_s = s, i, s
            for n in neighbours.get(i, ()):
                if mode == 0:
                    if n not in share:
                        continue
                    ns = self.reloc_score.get(n, F32(0.0))
                else:
                    if n not in scored:
                        continue
                    ns = scored[n]
                acc = F32(acc + ns)
                if ns > best_s:
                    best, best_s = n, ns
            acc_best.append((acc, best))
            best_acc = max(best_acc, acc)
        keep = F32(0.75) * best_acc
        out = []
        for acc, best in acc_best:
            if acc > keep and best not in out:
                out.append(best)
        return [i for i, _ in entries], [s for _, s in entries], out


class Both:
    """The oracle and the model side by side; every query asserts that they agree and returns the oracle's result."""

    def __init__(self, n_words, neighbours=None):
        self.o, self.m, self.nb = okl.KeyFrameDatabase(n_words), Model(n_words), neighbours or {}
        self.o.set_neighbours(self.nb)

    def set_neighbours(self, nb):
        self.nb = nb
        self.o.set_neighbours(nb)

    def add(self, i, bow):
        r = self.o.add(i, bow)
        assert r == self.m.add(i, bow)
        return r

    def erase(self, i):
        self.o.erase(i)
        self.m.erase(i)

    def clear(self):
        self.o.clear()
        self.m.clear()

    def query(self, mode, bow, min_score=0.0, connected=()):
        sid, ssc, cid = self.o.query(mode, bow, min_score, connected)
        mid, msc, mcid = self.m.query(mode, bow, min_score, set(connected), self.nb)
        assert sid.tolist() == mid and cid.tolist() == mcid
        np.testing.assert_array_equal(ssc, np.array(msc, np.float32))
        return sid.tolist(), ssc, cid.tolist()


def bow(words, values=None):
    w = np.array(sorted(words), np.uint32)
    v = np.full(len(w), 1.0 / max(len(w), 1)) if values is None else np.asarray(values, np.float64)
    return w, v


def random_bow(rng, n_words, n):
    w = np.sort(rng.choice(n_words, n, replace=False)).astype(np.uint32)
    v = rng.random(n)
    return w, v / v.sum()


def test_l1_score_matches_reading():
    rng = np.random.default_rng(0)
    for _ in range(200):
        a, b = random_bow(rng, 300, int(rng.integers(0, 80))), random_bow(rng, 300, int(rng.integers(0, 80)))
        assert okl.l1_score(a, b) == l1(a, b)
    a = random_bow(rng, 300, 50)
    assert okl.l1_score(a, a) == l1(a, a) and abs(l1(a, a) - 1.0) < 1e-12


@pytest.mark.parametrize("seed", range(6))
def test_random_databases_agree(seed):
    """Random databases on a small vocabulary (many shared words), random covisibility tables, consecutive reloc
    queries (stale scores), loop queries with connected sets and min scores, erase / re-add / clear in between."""
    rng = np.random.default_rng(seed)
    n_words = int(rng.choice([40, 200, 1000]))
    ids = rng.choice(10 ** 6, 120, replace=False).tolist()
    bows = {i: random_bow(rng, n_words, int(rng.integers(1, min(60, n_words)))) for i in ids}
    nb = {i: [int(x) for x in rng.choice(ids + [10 ** 7], int(rng.integers(0, 11)), replace=False)] for i in ids}
    d = Both(n_words, nb)
    for i in ids[:80]:
        assert d.add(i, bows[i]) == 0
    assert d.add(ids[0], bows[ids[0]]) == -1
    for step in range(40):
        op = rng.integers(0, 10)
        if op == 0:
            for i in rng.choice(ids, 5).tolist():
                d.erase(i)
        elif op == 1:
            for i in rng.choice(ids, 8).tolist():
                if i not in d.m.live:
                    d.add(i, bows[i])
        elif op == 2 and step == 20:
            d.clear()
            for i in ids[40:]:
                d.add(i, bows[i])
        q = random_bow(rng, n_words, int(rng.integers(0, 60)))
        if rng.random() < 0.3:  # a re-rendered database keyframe: many shared words
            q = bows[int(rng.choice(ids))]
        if rng.random() < 0.5:
            d.query(0, q)
        else:
            conn = rng.choice(ids, int(rng.integers(0, 10)), replace=False).tolist()
            d.query(1, q, float(rng.random() * 0.3), conn)
    assert d.o.size() == len(d.m.live)


# ---- one hand-built case per rule


def test_truncation():
    """max 7 common words -> minCommonWords = int(7 * 0.8f) = 5: 6 words are scored, 5 are not."""
    d = Both(100)
    d.add(1, bow(range(7)))
    d.add(2, bow(range(6)))
    d.add(3, bow(range(5)))
    sid, _, cid = d.query(0, bow(range(7)))
    assert sid == [1, 2] and cid == [1, 2]


def test_strict_greater_best_keyframe():
    """Two keyframes with equal scores, each the other's neighbour: pBestKF stays the entry itself."""
    d = Both(100, {1: [2], 2: [1]})
    d.add(1, bow([1, 2, 3]))
    d.add(2, bow([1, 2, 3]))
    sid, ssc, cid = d.query(0, bow([1, 2, 3, 4]))
    assert sid == [1, 2] and ssc[0] == ssc[1] and cid == [1, 2]


def test_shared_best_keyframe_is_listed_once():
    d = Both(100, {1: [3], 2: [3]})
    d.add(1, bow([1, 2, 3, 4, 50]))
    d.add(2, bow([1, 2, 3, 4, 51]))
    d.add(3, bow([1, 2, 3, 4]))
    sid, ssc, cid = d.query(0, bow([1, 2, 3, 4]))
    assert sid == [1, 2, 3] and ssc[2] > ssc[0] and cid == [3]


def test_stale_reloc_score_and_initial_zero():
    """Keyframe 9 shares one word with the second query but is not scored: it contributes the score the first query
    gave it, which beats the entry's own score.  Before any query scored it, it contributes 0."""
    d = Both(100, {1: [9]})
    d.add(1, bow([1, 2, 3, 4, 5, 6, 7, 8], [0.05] * 8))
    d.add(9, bow([1, 20, 21, 22]))
    q2 = bow([1, 2, 3, 4, 5, 6, 7, 8])
    sid, ssc, cid = d.query(0, q2)  # 9 shares word 1 but was never scored: initial 0.0f
    assert sid == [1] and cid == [1]
    sid, ssc9, _ = d.query(0, bow([1, 20, 21, 22]))  # scores 9 with 1.0
    assert 9 in sid
    sid, ssc, cid = d.query(0, q2)  # 9 is stale now: acc = s1 + 1.0, best = 9
    assert sid == [1] and cid == [9]


def test_order_after_erase_and_readd():
    d = Both(100)
    d.add(1, bow([1, 2]))
    d.add(2, bow([1, 2]))
    d.add(3, bow([2, 3]))
    assert d.query(0, bow([1, 2, 3]))[0] == [1, 2, 3]
    d.erase(1)
    d.add(1, bow([1, 2]))
    assert d.query(0, bow([1, 2, 3]))[0] == [2, 1, 3]
    d.erase(77)  # unknown id: no-op
    assert d.o.size() == 3


def test_loop_connected_and_min_score():
    d = Both(100)
    d.add(1, bow([1, 2, 3]))
    d.add(2, bow([1, 2, 3]))
    d.add(3, bow([1, 2, 3, 4, 5, 6], [0.5, 0.1, 0.1, 0.1, 0.1, 0.1]))
    q = bow([1, 2, 3])
    assert d.query(1, q, 0.0, [])[0] == [1, 2, 3]
    assert d.query(1, q, 0.0, [1])[0] == [2, 3]          # a connected keyframe is never listed
    sid, ssc, cid = d.query(1, q, 0.6, [2])              # keyframe 3 scores below 0.6: scored, not listed
    assert sid == [1] and cid == [1]


def test_query_keyframe_in_database():
    d = Both(100, {5: [6], 6: [5]})
    d.add(5, bow([1, 2, 3]))
    d.add(6, bow([2, 3, 4]))
    sid, ssc, cid = d.query(1, bow([1, 2, 3]), 0.1, [6])
    assert sid == [5] and ssc[0] == np.float32(1.0) and cid == [5]


def test_empty_cases():
    d = Both(100)
    assert d.query(0, bow([1, 2]))[2] == []
    d.add(1, bow([5, 6]))
    assert d.query(0, bow([]))[2] == [] and d.query(1, bow([1, 2]), 0.0)[2] == []
    assert d.add(2, bow([5, 100])) == -1                  # word id out of range
    assert d.add(3, (np.array([6, 5], np.uint32), np.ones(2))) == -1  # not ascending
