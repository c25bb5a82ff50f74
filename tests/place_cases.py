"""Hand-built inputs for the place-recognition scan, one rule each, on the edges of the scan's layout.

Every case is a small pool of descriptors plus a row map, db = pool[row_of], so place_ref.top2_pooled is exact.  The
background is random descriptors, about 128 bits from every query; the rows a case is about are planted at exact
distances (chosen bits of the query flipped) well below that.  A case asserts on the host, when it is built, that it
sits on its edge: the layout predicates under place_ref.scan_layout for the given SM count, and the reference's
answer for every planted query.  build(name, n_sm) rebuilds a case from its seed.
"""
from dataclasses import dataclass, field

import numpy as np

import place_ref as R

TH = 50  # TH_LOW, the vote threshold the benchmark and the product use


@dataclass
class Case:
    name: str
    rule: str
    q: np.ndarray
    pool: np.ndarray
    row_of: np.ndarray
    desc_per_kf: int = 8
    first_kf: int = 0
    th: int = TH
    expect: dict = field(default_factory=dict)  # query -> ((d0, i0), (d1, i1)), in-shard row indices

    @property
    def db(self):
        return self.pool[self.row_of]

    @property
    def n_kf(self):
        return (len(self.row_of) + self.desc_per_kf - 1) // self.desc_per_kf

    @property
    def first_index(self):
        return self.first_kf * self.desc_per_kf

    def reference(self):
        return R.top2_pooled(self.q, self.pool, self.row_of, self.first_index)


class _Builder:
    def __init__(self, name, rule, ndb, nq, seed, n_bg=64, **kw):
        self.rng = np.random.default_rng(seed)
        self.name, self.rule, self.kw = name, rule, kw
        self.q = self.rng.integers(0, 256, (nq, 32), dtype=np.uint8)
        self.pool = list(self.rng.integers(0, 256, (n_bg, 32), dtype=np.uint8))
        self.row_of = self.rng.integers(0, n_bg, ndb).astype(np.int64)
        self.used = set()
        self.reserved = set()
        self.expect = {}
        self.next_q = 0

    def query(self):
        """The next query not yet given a planted answer."""
        qi = self.next_q
        self.next_q += 1
        return qi

    def entry(self, desc):
        self.pool.append(np.asarray(desc, np.uint8))
        return len(self.pool) - 1

    def near(self, qi, dist):
        bits = np.unpackbits(self.q[qi])
        bits[self.rng.choice(256, dist, replace=False)] ^= 1
        return self.entry(np.packbits(bits))

    def put(self, rows, e):
        for r in rows:
            r = int(r)
            assert 0 <= r < len(self.row_of) and r not in self.used, (self.name, r)
            self.used.add(r)
            self.row_of[r] = e

    def reserve(self, rows):
        """Rows a case will plant later: free_row keeps off them."""
        self.reserved.update(int(r) for r in rows)

    def free_row(self):
        while True:
            r = int(self.rng.integers(0, len(self.row_of)))
            if r not in self.used and r not in self.reserved:
                return r

    def free_rows(self, k):
        rows = set()
        while len(rows) < k:
            rows.add(self.free_row())
        return sorted(rows)

    def best_tie(self, rows, dist=10, qi=None):
        """rows (ascending) hold one descriptor at `dist` from a query: the two lowest are its best and second."""
        qi = self.query() if qi is None else qi
        self.put(rows, self.near(qi, dist))
        self.expect[qi] = ((dist, rows[0]), (dist, rows[1]))
        return qi

    def second_tie(self, rows, dist=12, qi=None):
        """A strictly better row elsewhere, and `rows` tied for the second place: the lowest of them wins it."""
        qi = self.query() if qi is None else qi
        b = self.free_row()
        self.put([b], self.near(qi, dist - 7))
        self.put(rows, self.near(qi, dist))
        self.expect[qi] = ((dist - 7, b), (dist, rows[0]))
        return qi

    def done(self):
        c = Case(self.name, self.rule, self.q, np.stack(self.pool), self.row_of, expect=self.expect, **self.kw)
        d, i = c.reference()
        for qi, ((d0, i0), (d1, i1)) in self.expect.items():
            got = ((d[qi, 0], i[qi, 0] - c.first_index if i[qi, 0] >= 0 else -1),
                   (d[qi, 1], i[qi, 1] - c.first_index if i[qi, 1] >= 0 else -1))
            assert got == ((d0, i0), (d1, i1)), (self.name, qi, got, self.expect[qi])
        return c


def _lays(ndb, nq, n_sm):
    return {k: R.scan_layout(k, ndb, nq, n_sm) for k in R.KINDS}


# ---------------------------------------------------------------------------------------------------- the cases
def _ties(n_sm, triples):
    """Two (or three) rows tied at every position where a kernel merges partial results: the halves of a packed TMEM
    register, the two 32-column loads of a tile, tiles of every pair of accumulator groups, the imma quad columns, the
    imma and POPC tile edges, and slice cuts of every kernel.  Each position is tied once for the best and once (768
    rows on, which keeps the umma group and every kernel's column, or at another slice cut) for the second best."""
    nq = 128
    ndb = 4096 * n_sm + 37
    L = _lays(ndb, nq, n_sm)
    u = L["umma"]
    assert all(l.qblocks == 1 for l in L.values())
    assert u.tiles_per_cta >= 31 and L["imma"].tiles_per_cta >= 2 and L["popc"].tiles_per_cta >= 2, L
    if triples:
        sets = [(0, 1, 2), (63, 64, 128), (129, 193, 257), (128 + 60, 192 + 61, 256 + 62, 320 + 63)]
        assert [R.group(u, r) for r in sets[2]] == [2, 0, 1]
    else:
        sets = [
            (0, 1), (44, 45), (4 * 64 + 62, 4 * 64 + 63),         # adjacent columns 2j / 2j+1 (one packed register)
            (31, 32), (63, 64),                                   # the two 32-column loads; the tile edge
            (10, 64 + 10), (64 + 40, 128 + 40), (20, 128 + 20),   # groups 0/1, 1/2, 0/2
            (128 + 50, 192 + 50), (64 + 50, 192 + 51),            # group 2, group 1 before a later tile of group 0
            (5 * 64 + 3, 6 * 64 + 3),                             # group 2 before group 0, second round of tiles
            (18, 19), (34, 42), (49, 50),                         # imma: 2t / 2t+1, n0 / n0+8, across quad lanes
            (127, 128), (255, 256),                               # imma tile edges; the POPC tile edge
        ]
        assert [(R.group(u, a), R.group(u, b)) for a, b in sets[5:11]] == [(0, 1), (1, 2), (0, 2), (2, 0), (1, 0), (2, 0)]
        assert [R.in_tile(u, r) for r in (31, 32, 63, 64)] == [31, 32, 63, 0]
        assert [R.in_tile(L["imma"], r) % 8 for r in (18, 19, 34, 42, 49, 50)] == [2, 3, 2, 2, 1, 2]
        assert R.in_tile(L["imma"], 128) == 0 and R.in_tile(L["popc"], 256) == 0 and R.in_tile(L["popc"], 255) == 255
    shift = 768  # 12 umma tiles (4 rounds of the 3 groups), 6 imma tiles, 3 POPC tiles
    assert all(R.slice_of(u, r + shift) == 0 for t in sets for r in t)
    cuts = {}  # kind -> [(slice, rows straddling its first row)]
    for kind, lay in L.items():
        starts = R.slice_starts(lay)
        assert len(starts) >= 6, (kind, lay)
        w = len(sets[0])
        sl = sorted({1, 2, len(starts) // 2, len(starts) // 2 + 1, len(starts) - 2, len(starts) - 1})
        cuts[kind] = [tuple(range(starts[s] - 1, starts[s] - 1 + w)) for s in sl]
        for s, c in zip(sl, cuts[kind]):
            assert R.slice_of(lay, c[0]) + 1 == R.slice_of(lay, c[1]) == s
    b = _Builder("three_tied" if triples else "ties_positions",
                 "of three or more tied rows only the two lowest appear" if triples else
                 "ties for best and second best go to the lower index", ndb, nq, 11 if triples else 10)
    plan = [(list(t), [r + shift for r in t]) for t in sets]
    taken = {r for x, y in plan for r in x + y}
    for kind in L:  # cuts of one kernel that are not already in the plan: best tie at one, second at the next
        c = [list(x) for x in cuts[kind] if not set(x) & taken]
        assert len(c) >= 2, (kind, cuts[kind])
        taken.update(r for x in c for r in x)
        plan += [(c[i], c[i + 1] if i + 1 < len(c) else None) for i in range(0, len(c), 2)]
    b.reserve(taken)
    for x, y in plan:
        b.best_tie(x)
        if y:
            b.second_tie(y)
    assert b.next_q <= nq
    return b.done()


def _query_positions(n_sm, nq):
    """Queries at the first row of A tile 0, the last / first of A tiles 0 / 1 (127 / 128), and the last / first of
    query blocks (255 / 256), and the last query, at nq on both sides of those edges."""
    ndb = 5000
    b = _Builder(f"query_pos_nq{nq}", "query rows at A-tile and query-block edges", ndb, nq, 20 + nq)
    for qi in sorted({p for p in (0, 127, 128, 255, 256, nq - 1) if p < nq}):
        b.best_tie(b.free_rows(3), dist=9 + qi % 7, qi=qi)
    for lay in _lays(ndb, nq, n_sm).values():
        assert lay.qblocks == (nq + lay.qper - 1) // lay.qper
    return b.done()


def _chunk_filter(n_sm, g):
    """db_top2_umma_kernel skips a 32-column chunk unless some lane of the warp sees a key strictly below its running
    second-best distance.  All 32 queries of warp 0 get a best at 20 and a second at 30 in the first tile of group g;
    then later rows at exactly 30 (must not replace), at 29 (must replace; alone in its chunk for the whole warp), and
    at 19 (new best), in the same tile, in a later tile of the group, and in another group."""
    nq = 32
    ndb = 64 * 24 * n_sm + 17
    u = R.scan_layout("umma", ndb, nq, n_sm)
    assert u.tiles_per_cta >= 12, u
    b = _Builder(f"chunk_filter_g{g}", "chunk filter: strictly below the running second best", ndb, nq, 30 + g)
    T = lambda t, c: 64 * t + c  # noqa: E731  row of column c in local tile t of slice 0
    base = {}
    for m in range(3, 32):  # baseline of queries 3..31 in the first tile of group g
        base[m] = (T(g, 2 * (m - 3)), T(g, 2 * (m - 3) + 1))
    for m in range(3):      # queries 0..2 get theirs in the next tile of the group, with same-tile targets
        base[m] = (T(g + 3, 2 * m), T(g + 3, 2 * m + 1))
    for m, (r0, r1) in base.items():
        b.put([r0], b.near(m, 20))
        b.put([r1], b.near(m, 30))
        b.expect[m] = ((20, r0), (30, r1))
    targets = {  # query: (row, distance)
        0: (T(g + 3, 10), 30), 1: (T(g + 3, 40), 29), 2: (T(g + 3, 50), 19),   # same tile
        3: (T(g + 6, 3), 30), 4: (T(g + 6, 40), 29), 5: (T(g + 9, 7), 19),     # later tiles of group g
        6: (T(g + 4, 5), 29), 7: (T(g + 4, 20), 30), 8: (T(g + 4, 50), 19),    # group g + 1
    }
    for m, (row, dist) in targets.items():
        b.put([row], b.near(m, dist))
        r0, r1 = base[m]
        b.expect[m] = {30: ((20, r0), (30, r1)), 29: ((20, r0), (29, row)), 19: ((19, row), (20, r0))}[dist]
    b.next_q = nq
    for m, (row, _) in targets.items():
        assert R.slice_of(u, row) == 0 and R.group(u, row) == ((g + 1) % 3 if m >= 6 else g)
    # query 4's row is alone in its chunk: no other (query of the warp, row of the chunk) is below 30
    c = b.done()
    row4 = targets[4][0]
    chunk = np.arange(row4 - row4 % 32, row4 - row4 % 32 + 32)
    d = R.hamming(c.q, c.pool[c.row_of[chunk]])
    d[4, chunk == row4] = 99
    assert d.min() >= 30 and R.in_tile(u, row4) >= 32
    return c


def _extremes(which):
    """Distances 0 and 256 as best and as second best; all-zero and all-one queries and rows, popcounts 1 and 255."""
    zeros, ones = np.zeros(32, np.uint8), np.full(32, 255, np.uint8)
    e7 = np.packbits(np.eye(256, dtype=np.uint8)[7])
    if which == "mixed":
        b = _Builder("dist_0_256_mixed", "distance 0 ties, popcount 1 / 255 neighbours", 70, 6, 40)
        b.q[:4] = [zeros, ones, e7, ~e7]
        z, o, p1, p255 = b.entry(zeros), b.entry(ones), b.entry(e7), b.entry(~e7)
        b.put([5, 66], z)
        b.put([7], o)
        b.put([9], p255)
        b.put([11], p1)
        b.expect = {0: ((0, 5), (0, 66)), 1: ((0, 7), (1, 9)), 2: ((0, 11), (1, 5)), 3: ((0, 9), (1, 7))}
    elif which == "256":
        b = _Builder("dist_256_only", "distance 256 as best and second best", 5, 4, 41, n_bg=1)
        b.pool = [ones]
        b.row_of[:] = 0
        b.q[:3] = [zeros, ones, e7]
        b.expect = {0: ((256, 0), (256, 1)), 1: ((0, 0), (0, 1)), 2: ((255, 0), (255, 1))}
    else:
        b = _Builder("dist_255_256", "distance 255 best, 256 second", 3, 3, 42, n_bg=1)
        b.pool = [ones, ~e7]
        b.row_of[:] = [0, 0, 1]
        b.q[:2] = [zeros, e7]
        b.expect = {0: ((255, 2), (256, 0)), 1: ((255, 0), (255, 1))}
    return b.done()


def _tail(T, r):
    """ndb = T m + r: the last tile of every kernel is partial.  An all-zero query against a database with no zero row:
    a padding row that is not masked would win at distance 0."""
    ndb = T * 5 + r
    b = _Builder(f"tail_{T}_{r}", "masked tail tile", ndb, 10, 50 + T + r)
    b.q[0] = 0
    b.q[1] = 255
    b.best_tie([ndb - r - 1, ndb - 1], dist=3, qi=2)  # the last full tile against the last row
    b.second_tie([ndb - r - 2, ndb - 2] if r >= 2 else [ndb - r - 3, ndb - r - 2], qi=3)
    c = b.done()
    d, _ = c.reference()
    assert (c.pool != 0).any(1).all() and d[0, 0] > 0
    assert all(ndb % R.scan_layout(k, ndb, 10, 148).tile != 0 for k in R.KINDS)
    return c


def _small(ndb):
    """Databases of 1 to 3 rows: the second best is missing for ndb = 1."""
    b = _Builder(f"small_ndb{ndb}", "tiny database, missing second best", ndb, 5, 60 + ndb, n_bg=2)
    b.q[0] = b.pool[b.row_of[0]]
    d, i = R.top2_dense(b.q, np.stack(b.pool)[b.row_of])
    assert (ndb == 1) == (i[:, 1] == -1).all()
    return b.done()


def _last_slice(n_sm, ntiles):
    """umma slices whose last one has 1, 2 or 3 tiles: accumulator groups without a tile."""
    nq = 40
    ndb = 2 * n_sm * 4 * 64
    while True:
        u = R.scan_layout("umma", ndb, nq, n_sm)
        if u.tiles_per_cta >= 4 and R.slice_tiles(u, u.parts - 1) == ntiles:
            break
        ndb += 64
    ndb -= 64 - 13  # the last tile holds 13 rows
    u = R.scan_layout("umma", ndb, nq, n_sm)
    assert R.slice_tiles(u, u.parts - 1) == ntiles and u.tiles_per_cta >= 4
    b = _Builder(f"last_slice_{ntiles}_tiles", "short last slice, empty accumulator groups", ndb, nq, 70 + ntiles)
    s = R.slice_starts(u)[-1]
    b.best_tie([s, ndb - 1])
    b.second_tie([s + 1, s + 2])
    b.best_tie([s - 1, s + 3])
    if ntiles > 1:
        b.best_tie([s + 64 + 5, ndb - 2])
        assert R.group(u, s + 64 + 5) == 1
    return b.done()


def _votes(th):
    """Votes: best exactly th and th + 1, desc_per_kf = 7 not dividing ndb, first_kf > 0, a best in the short last
    keyframe, several queries on one keyframe."""
    dpk, ndb = 7, 7 * 300 + 3
    b = _Builder(f"votes_th{th}", "vote: best <= th, inclusive", ndb, 12, 80 + th, desc_per_kf=dpk, first_kf=1234, th=th)
    b.best_tie([70, 71], dist=th)            # votes for keyframe 10
    b.best_tie([140, 900], dist=th + 1)      # no vote
    b.best_tie([2100, 2102], dist=0)         # the short last keyframe (3 rows)
    b.best_tie([0, 1], dist=max(th - 3, 0))  # keyframe 0
    b.best_tie([2, 3], dist=th)              # keyframe 0 again
    b.second_tie([700, 701], dist=th + 7)    # best at th (a row elsewhere), second above
    c = b.done()
    assert len(c.row_of) % dpk != 0 and c.first_kf > 0
    return c


def clamp(kind, n_sm):
    """db_scan keeps the in-slice index of the 32-bit keys to 20 bits: tiles_per_cta <= 2^20 / tile.  With one query
    block more than the SMs (umma) or than 4 x the SMs (imma) there is one slice per query block before the clamp, so
    2^20 + 3 x 64 + 5 rows need it.  Ties straddle rows 2^20 - 1 / 2^20 and a best sits at in-slice index 2^20 - 1;
    the planted queries are the first two and the last two, in the last query block."""
    nq = 256 * (1 if kind == "umma" else 4) * n_sm + 1
    ndb = (1 << 20) + 3 * 64 + 5
    lay = R.scan_layout(kind, ndb, nq, n_sm)
    assert lay.parts == 2 and lay.slice_rows == 1 << 20 and lay.tiles > lay.tiles_per_cta, lay
    M = 1 << 20
    b = _Builder(f"clamp_{kind}", "20-bit in-slice index", ndb, nq, 90)
    b.reserve([M - 3, M - 2, M - 1, M, M + 1, M + 2, ndb - 1])
    b.best_tie([M - 1, M], qi=0)                       # best at in-slice index 2^20 - 1, second at slice 1 row 0
    b.best_tie([M + 1, ndb - 1], qi=1)                 # both in the second slice, the last row among them
    b.second_tie([M - 2, M + 2], qi=nq - 2)
    b.put([M - 3], b.near(nq - 1, 4))
    c = b.done()
    d, i = c.reference()
    assert d[nq - 1, 0] == 4 and i[nq - 1, 0] == M - 3
    assert R.slice_of(lay, M - 1) == 0 and R.slice_of(lay, M) == 1 and (M - 1) % lay.slice_rows == M - 1
    return c


_BUILDERS = {"ties_positions": lambda n: _ties(n, False), "three_tied": lambda n: _ties(n, True)}
for _nq in (1, 127, 128, 129, 255, 256, 257):
    _BUILDERS[f"query_pos_nq{_nq}"] = lambda n, nq=_nq: _query_positions(n, nq)
for _g in range(3):
    _BUILDERS[f"chunk_filter_g{_g}"] = lambda n, g=_g: _chunk_filter(n, g)
for _w in ("mixed", "256", "255"):
    _BUILDERS[{"mixed": "dist_0_256_mixed", "256": "dist_256_only", "255": "dist_255_256"}[_w]] = lambda n, w=_w: _extremes(w)
for _T in (64, 128, 256):
    for _r in (1, 31, 32, 33, 63):
        _BUILDERS[f"tail_{_T}_{_r}"] = lambda n, T=_T, r=_r: _tail(T, r)
for _n in (1, 2, 3):
    _BUILDERS[f"small_ndb{_n}"] = lambda n, k=_n: _small(k)
    _BUILDERS[f"last_slice_{_n}_tiles"] = lambda n, k=_n: _last_slice(n, k)
for _th in (TH, 0):
    _BUILDERS[f"votes_th{_th}"] = lambda n, th=_th: _votes(th)

NAMES = sorted(_BUILDERS)


def build(name, n_sm):
    c = _BUILDERS[name](n_sm)
    assert c.name == name
    return c
