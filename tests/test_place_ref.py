"""place_ref, the independent reading of the place-recognition scan, against the oracle and against itself, and the
edge assertions of every place_cases case at several SM counts (CPU only)."""
import numpy as np
import pytest
import torch

import place_cases as P
import place_ref as R


def _random_and_tied(seed, nq, ndb, npool=None):
    rng = np.random.default_rng(seed)
    q = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    pool = rng.integers(0, 256, (npool or ndb, 32), dtype=np.uint8)
    if npool:  # tie-heavy: a few descriptors, some of them near a query, repeated over the rows
        pool[: min(npool, nq)] = q[: min(npool, nq)] ^ rng.integers(0, 2, (min(npool, nq), 32), dtype=np.uint8)
        row_of = rng.integers(0, npool, ndb)
    else:
        row_of = np.arange(ndb)
    return q, pool, row_of


SHAPES = [(40, 1, None), (40, 2, None), (40, 3, None), (33, 700, None), (33, 700, 5), (64, 3000, 3), (17, 257, 1)]


@pytest.mark.parametrize("nq,ndb,npool", SHAPES)
def test_dense_equals_oracle(oracle, nq, ndb, npool):
    q, pool, row_of = _random_and_tied(nq + ndb, nq, ndb, npool)
    db = pool[row_of]
    q[0] = 0
    o = oracle.bruteforce_top2(q, db)
    d, i = R.top2_dense(q, db)
    # the oracle reports a missing entry as distance 257, index -1
    np.testing.assert_array_equal(np.stack([d[:, 0], i[:, 0], d[:, 1], i[:, 1]], 1),
                                  np.where(o == 257, -1, o))


@pytest.mark.parametrize("first_index", [0, 1234 * 7])
@pytest.mark.parametrize("nq,ndb,npool", SHAPES)
def test_pooled_and_gemm_equal_dense(nq, ndb, npool, first_index):
    q, pool, row_of = _random_and_tied(nq * ndb, nq, ndb, npool)
    q[1] = 255
    d, i = R.top2_dense(q, pool[row_of], first_index)
    for name, (d2, i2) in {"pooled": R.top2_pooled(q, pool, row_of, first_index),
                           "gemm": R.top2_gemm(q, pool[row_of], first_index, chunk=256)}.items():
        np.testing.assert_array_equal(d2, d, err_msg=name)
        np.testing.assert_array_equal(i2, i, err_msg=name)
    assert (i[:, 1] == -1).all() == (ndb == 1)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_votes_sum_over_partition_equals_votes_from_global(world):
    from swarmmap_b200 import place
    rng = np.random.default_rng(world)
    dpk, nkf = 7, 61
    ndb = dpk * nkf - 2
    nq = 300
    d = rng.integers(0, 257, nq)
    d[:20] = 50
    d[20:40] = 51
    i = rng.integers(0, ndb, nq)
    i[:5] = ndb - 1
    i[5:10] = -1
    merged = torch.from_numpy(np.stack([R.pack(d, i), R.pack(d, i)], 1))
    total = np.zeros(nkf, np.int64)
    for f, n in place.partition(nkf, world):
        rows = min((f + n) * dpk, ndb) - f * dpk
        sh = place.PlaceShard(np.zeros((rows, 32), np.uint8), dpk, f, local_topk=lambda *a: None)
        mine = R.votes(merged[:, 0].numpy(), 50, dpk, f, sh.n_kf)
        np.testing.assert_array_equal(mine, sh.votes_from_global(merged, 50).numpy())
        total[f:f + sh.n_kf] += mine
    np.testing.assert_array_equal(total, R.votes(merged[:, 0].numpy(), 50, dpk, 0, nkf))
    assert total.sum() == ((d <= 50) & (i >= 0)).sum()


@pytest.mark.parametrize("n_sm", [148, 132, 160])
@pytest.mark.parametrize("name", P.NAMES)
def test_case_sits_on_its_edge(name, n_sm):
    c = P.build(name, n_sm)  # asserts the layout predicates and the reference's answer for every planted query
    assert c.name == name and len(c.q) > 0


@pytest.mark.parametrize("n_sm", [148, 132, 160])
@pytest.mark.parametrize("kind", ["umma", "imma"])
def test_clamp_case_sits_on_its_edge(kind, n_sm):
    c = P.clamp(kind, n_sm)
    assert R.scan_layout(kind, len(c.row_of), len(c.q), n_sm).parts == 2


def test_scan_layout_of_the_benchmark():
    """World 1 at 148 SMs: 37 umma slices of 691 904 rows, as the README's config-5 row states."""
    lay = R.scan_layout("umma", 100000 * 256, 2000, 148)
    assert (lay.parts, lay.slice_rows) == (37, 691904)
