"""The config-5 place-recognition scan (db_top2_umma_kernel, db_top2_mma_kernel, db_top2_kernel, db_merge_kernel,
db_merge_peers_kernel and db_scan's slices) against place_ref, an independent reading: every hand-built case of
place_cases on each kernel, the 20-bit in-slice clamp, and every query of the benchmark's own config-5 input at
world 1, 2 and 8.  Keys and votes must be equal."""
import ctypes as C
import functools
import os

import numpy as np
import pytest
import torch

import place_cases as P
import place_ref as R

pytestmark = pytest.mark.gpu

TH = 50


@pytest.fixture(scope="module")
def n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


@functools.lru_cache(maxsize=None)
def _case(name, n_sm):
    c = P.clamp(name[len("clamp_"):], n_sm) if name.startswith("clamp_") else P.build(name, n_sm)
    return c, c.reference()


def _query(c, k, path):
    """(keys, votes) of one shard scan + merge, through PlaceShard (swm_db_create_device) or the host-array create."""
    from swarmmap_b200 import _lib, place
    if path == "device":
        sh = place.PlaceShard(c.db, c.desc_per_kf, c.first_kf)
        keys, votes = sh.query_local(torch.from_numpy(c.q), k, c.th)
        torch.cuda.synchronize()
        sh.close()
        return keys, votes.cpu().numpy()
    lib = _lib.load()
    db = np.ascontiguousarray(c.db)
    h = C.c_void_p()
    assert lib.swm_db_create(0, _lib.ptr(db), len(db), c.desc_per_kf, c.first_kf, C.byref(h)) == 0
    dq = torch.from_numpy(c.q).cuda()
    keys = torch.zeros((len(c.q), k), dtype=torch.int64, device="cuda")
    votes = torch.zeros(c.n_kf, dtype=torch.int32, device="cuda")
    rc = lib.swm_db_query_device(h, dq.data_ptr(), len(c.q), k, keys.data_ptr(), votes.data_ptr(), c.th, None)
    torch.cuda.synchronize()
    lib.swm_db_destroy(h)
    assert rc == 0
    return keys, votes.cpu().numpy()


def _assert_keys(keys, ref, k, what=""):
    gd, gi = R.unpack(keys)
    d, i = ref
    bad = np.nonzero((gd != d[:, :k]).any(1) | (gi != i[:, :k]).any(1))[0]
    assert len(bad) == 0, (f"{what}: {len(bad)} queries differ, first {bad[:5].tolist()}: "
                           f"device {list(zip(gd[bad[0]], gi[bad[0]]))} ref {list(zip(d[bad[0], :k], i[bad[0], :k]))}")


def _ref_votes(ref, th, dpk, first_kf, n_kf):
    return R.votes(R.pack(ref[0][:, 0], ref[1][:, 0]), th, dpk, first_kf, n_kf)


# ------------------------------------------------------------------------------------------ a. every case
@pytest.mark.parametrize("path", ["device", "host"])
@pytest.mark.parametrize("k", [1, 2])
@pytest.mark.parametrize("kernel", R.KINDS)
@pytest.mark.parametrize("name", P.NAMES)
def test_case(swm, monkeypatch, n_sm, name, kernel, k, path):
    monkeypatch.setenv("SWM_DB_KERNEL", kernel)
    c, ref = _case(name, n_sm)
    keys, votes = _query(c, k, path)
    _assert_keys(keys, ref, k, f"{name} ({c.rule})")
    np.testing.assert_array_equal(votes, _ref_votes(ref, c.th, c.desc_per_kf, c.first_kf, c.n_kf))


# ------------------------------------------------------------------------------------------ b. the 20-bit clamp
@pytest.mark.parametrize("kernel", ["umma", "imma"])
def test_in_slice_index_clamp(swm, monkeypatch, n_sm, kernel):
    """2^20 + 197 rows and one query block more than the kernel's slices: db_scan must cut a second slice at 2^20."""
    monkeypatch.setenv("SWM_DB_KERNEL", kernel)
    c, ref = _case(f"clamp_{kernel}", n_sm)
    keys, votes = _query(c, 2, "device")
    _assert_keys(keys, ref, 2, c.name)
    np.testing.assert_array_equal(votes, _ref_votes(ref, c.th, c.desc_per_kf, c.first_kf, c.n_kf))


# ------------------------------------------------------------------------------------------ c. the benchmark's input
NQ, DPK, NKF = 2000, 256, 100000


def bench_place_inputs(world, rank):
    """workload_place's inputs for one rank, replayed draw for draw (bench.py lines 795-813): queries from a device
    generator seeded 99, the shard from one seeded 990 + rank, then every 100th keyframe overwritten by noisy copies
    of 256 consecutive queries in keyframe order."""
    from swarmmap_b200 import place
    dev = torch.device("cuda", 0)
    parts = place.partition(NKF, world)
    first_kf, n_kf = parts[rank]
    gq = torch.Generator(device=dev)
    gq.manual_seed(99)
    q = torch.randint(0, 256, (NQ, 32), dtype=torch.uint8, device=dev, generator=gq)
    gen = torch.Generator(device=dev)
    gen.manual_seed(990 + rank)
    db = torch.randint(0, 256, (n_kf * DPK, 32), dtype=torch.uint8, device=dev, generator=gen)
    planted = [kf for kf in range(first_kf, first_kf + n_kf) if kf % 100 == 0]
    for kf in planted:
        j0 = (kf * 7) % (NQ - DPK)
        flips = torch.rand((DPK, 256), device=dev, generator=gen) < 0.10
        bits = torch.zeros((DPK, 32), dtype=torch.uint8, device=dev)
        for bit in range(8):
            bits |= (flips[:, bit::8].to(torch.uint8) << bit)
        lo = (kf - first_kf) * DPK
        db[lo:lo + DPK] = q[j0:j0 + DPK] ^ bits
    return q, db, first_kf, n_kf


@functools.lru_cache(maxsize=None)
def _bench_world(world):
    shards = [bench_place_inputs(world, r) for r in range(world)]
    q = shards[0][0]
    full = torch.cat([s[1] for s in shards]) if world > 1 else shards[0][1]
    ref = R.top2_gemm(q, full)
    del full
    torch.cuda.empty_cache()
    return q, [(db, f, n) for _, db, f, n in shards], ref


@pytest.mark.parametrize("kernel", R.KINDS)
def test_bench_world1_every_query(swm, monkeypatch, kernel):
    from swarmmap_b200 import place
    monkeypatch.setenv("SWM_DB_KERNEL", kernel)
    q, ((db, first_kf, n_kf),), ref = _bench_world(1)
    sh = place.PlaceShard(db, DPK, first_kf)
    keys, votes = sh.query(q, 2, TH)
    torch.cuda.synchronize()
    _assert_keys(keys, ref, 2, "world 1")
    np.testing.assert_array_equal(votes.cpu().numpy(), _ref_votes(ref, TH, DPK, first_kf, n_kf))
    assert (ref[0][:, 0] <= TH).mean() > 0.8  # the planted keyframes are found


def _merge_gathered(shards, q, k):
    """Each shard's local (nq, k) block stacked as all_gather_into_tensor lays them out, merged on every rank."""
    from swarmmap_b200 import _lib
    lib = _lib.load()
    gathered = torch.stack([s.query_local(q, k, TH)[0] for s in shards], 0).contiguous()
    out = []
    for s in shards:
        merged = torch.empty((len(q), k), dtype=torch.int64, device="cuda")
        votes = torch.zeros(s.n_kf, dtype=torch.int32, device="cuda")
        rc = lib.swm_db_merge_gathered(s._h, gathered.data_ptr(), len(shards), len(q), k, merged.data_ptr(),
                                       votes.data_ptr(), TH, None)
        assert rc == 0
        out.append((merged, votes))
    torch.cuda.synchronize()
    return out


def test_bench_world8_every_query(swm):
    from swarmmap_b200 import place
    q, parts, ref = _bench_world(8)
    shards = [place.PlaceShard(db, DPK, f) for db, f, _ in parts]
    for r, (merged, votes) in enumerate(_merge_gathered(shards, q, 2)):
        _assert_keys(merged, ref, 2, f"world 8 rank {r}")
        np.testing.assert_array_equal(votes.cpu().numpy(), _ref_votes(ref, TH, DPK, parts[r][1], parts[r][2]))


def _peers(shards, q, k):
    """query_peers with every rank on its own stream of one GPU, all enqueued before any result is read."""
    for sh in shards:
        sh.enable_peers(nq_max=len(q), same_process=shards)
    streams = [torch.cuda.Stream() for _ in shards]
    outs = []
    for r, sh in enumerate(shards):
        with torch.cuda.stream(streams[r]):
            outs.append(sh.query_peers(q, k, TH))
    torch.cuda.synchronize()
    return outs


def test_bench_world2_peers_every_query(swm):
    from swarmmap_b200 import place
    if os.environ.get("CUDA_LAUNCH_BLOCKING") == "1":
        pytest.skip("the ranks' kernels wait for each other: they cannot run with serialised launches")
    q, parts, ref = _bench_world(2)
    shards = [place.PlaceShard(db, DPK, f) for db, f, _ in parts]
    for r, (merged, votes) in enumerate(_peers(shards, q, 2)):
        _assert_keys(merged, ref, 2, f"world 2 rank {r}")
        np.testing.assert_array_equal(votes.cpu().numpy(), _ref_votes(ref, TH, DPK, parts[r][1], parts[r][2]))


# ------------------------------------------------------------------------------------------ d. pooled background
def _pooled_bench_shape(n_sm):
    """The benchmark's shape (2000 queries, 100 000 keyframes x 256) over a pool of 65 536 random descriptors, with ties
    planted across every slice cut of the world-1 umma layout and every cut of the 8-rank partition: at each cut one
    query has its best tied on the two rows that straddle it, another its second best on the next two."""
    from swarmmap_b200 import place
    rng = np.random.default_rng(5)
    ndb = NKF * DPK
    q = rng.integers(0, 256, (NQ, 32), dtype=np.uint8)
    pool = [rng.integers(0, 256, (65536, 32), dtype=np.uint8)]
    row_of = torch.randint(0, 65536, (ndb,), generator=torch.Generator().manual_seed(6), dtype=torch.int64)
    lay = R.scan_layout("umma", ndb, NQ, n_sm)
    cuts = sorted(set(R.slice_starts(lay)[1:]) | {f * DPK for f, _ in place.partition(NKF, 8)[1:]})
    expect, qi = {}, 0

    def near(j, dist):
        bits = np.unpackbits(q[j])
        bits[rng.choice(256, dist, replace=False)] ^= 1
        pool.append(np.packbits(bits)[None])
        return 65536 + len(pool) - 2

    for cut in cuts:
        e = near(qi, 10)
        row_of[[cut - 1, cut]] = e
        expect[qi] = ((10, cut - 1), (10, cut))
        e0, e1 = near(qi + 1, 5), near(qi + 1, 12)
        b = int(rng.integers(0, ndb - 4))
        while any(abs(b - c) < 4 for c in cuts):
            b = int(rng.integers(0, ndb - 4))
        row_of[b] = e0
        row_of[[cut - 2, cut + 1]] = e1
        expect[qi + 1] = ((5, b), (12, cut - 2))
        qi += 2
    pool = np.concatenate(pool)
    row_of = row_of.cuda()
    ref = R.top2_pooled(q, pool, row_of)
    for j, ((d0, i0), (d1, i1)) in expect.items():
        assert (ref[0][j, 0], ref[1][j, 0], ref[0][j, 1], ref[1][j, 1]) == (d0, i0, d1, i1), j
    db = torch.from_numpy(pool).cuda()[row_of]
    return torch.from_numpy(q).cuda(), db, ref


def test_pooled_bench_shape_world1_and_8(swm, n_sm):
    from swarmmap_b200 import place
    q, db, ref = _pooled_bench_shape(n_sm)
    full = place.PlaceShard(db, DPK, 0)
    keys, votes = full.query(q, 2, TH)
    torch.cuda.synchronize()
    _assert_keys(keys, ref, 2, "pooled world 1")
    np.testing.assert_array_equal(votes.cpu().numpy(), _ref_votes(ref, TH, DPK, 0, NKF))
    full.close()
    parts = place.partition(NKF, 8)
    shards = [place.PlaceShard(db[f * DPK:(f + n) * DPK], DPK, f) for f, n in parts]
    for r, (merged, v) in enumerate(_merge_gathered(shards, q, 2)):
        _assert_keys(merged, ref, 2, f"pooled world 8 rank {r}")
        np.testing.assert_array_equal(v.cpu().numpy(), _ref_votes(ref, TH, DPK, parts[r][0], parts[r][1]))


# ------------------------------------------------------------------------------------------ e. ties across shard cuts
def _cut_case(world):
    """A pooled database of 203 keyframes x 8 (and a short last one) cut by place.partition(203, world): at every cut
    a best tied across it (dist 10 <= TH: only the lower shard may vote), a second best tied across it, and three rows
    tied across it with a better best elsewhere."""
    from swarmmap_b200 import place
    dpk, nkf = 8, 203
    ndb = dpk * nkf - 3
    parts = place.partition(nkf, world)
    cuts = [f * dpk for f, _ in parts[1:]]
    b = P._Builder(f"cuts_{world}", "ties across shard cuts", ndb, 64, 100 + world, desc_per_kf=dpk)
    b.reserve([c + o for c in cuts for o in range(-3, 3)])
    for c in cuts:
        b.best_tie([c - 1, c])
        b.second_tie([c - 3, c + 1])
        b.second_tie([c - 2, c + 2])
    return b.done(), parts


@pytest.mark.parametrize("k", [1, 2])
@pytest.mark.parametrize("world", range(2, 9))
def test_ties_across_shard_cuts(swm, world, k):
    from swarmmap_b200 import place
    c, parts = _cut_case(world)
    ref = c.reference()
    db = c.db
    shards = [place.PlaceShard(db[f * c.desc_per_kf:min((f + n) * c.desc_per_kf, len(db))], c.desc_per_kf, f)
              for f, n in parts]
    total = np.zeros(c.n_kf, np.int64)
    for r, (merged, votes) in enumerate(_merge_gathered(shards, torch.from_numpy(c.q), k)):
        _assert_keys(merged, ref, k, f"{c.name} rank {r}")
        f, n = parts[r]
        np.testing.assert_array_equal(votes.cpu().numpy(), _ref_votes(ref, TH, c.desc_per_kf, f, shards[r].n_kf))
        total[f:f + shards[r].n_kf] += votes.cpu().numpy()
    np.testing.assert_array_equal(total, _ref_votes(ref, TH, c.desc_per_kf, 0, c.n_kf))
    if world <= 4 and os.environ.get("CUDA_LAUNCH_BLOCKING") != "1":  # all ranks' merge kernels wait on one GPU
        for r, (merged, votes) in enumerate(_peers(shards, torch.from_numpy(c.q), k)):
            _assert_keys(merged, ref, k, f"{c.name} peers rank {r}")
            np.testing.assert_array_equal(votes.cpu().numpy(),
                                          _ref_votes(ref, TH, c.desc_per_kf, parts[r][0], shards[r].n_kf))
