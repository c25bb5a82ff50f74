"""Second reading of the config-5 place-recognition scan: the top-2 of every query over a descriptor database, the
vote rule, and the slice arithmetic of db_scan.  numpy and torch only; it shares no code with the three scan kernels
(db_top2_umma_kernel in csrc/db_umma.cuh, db_top2_mma_kernel and db_top2_kernel in csrc/match.cu), with
db_merge_kernel, with the oracle or with swarmmap_b200.place.

Every top-2 function orders by (distance, global index) and returns (dist, index), each (nq, 2) int64, with a missing
entry as (-1, -1), the form place.unpack_keys gives for the device's packed keys (dist << 48 | global index).
"""
from collections import namedtuple

import numpy as np
import torch

IDX_BITS = 48
IDX_MASK = (1 << IDX_BITS) - 1
NONE = np.int64(np.iinfo(np.int64).max)  # sorts after every real key; unpacked as (-1, -1)


def _u64(a):
    return np.ascontiguousarray(a, np.uint8).reshape(-1, 32).view(np.uint64)


def hamming(q, db):
    """(nq, ndb) int64 Hamming distances between two small sets of 256-bit descriptors."""
    qa, da = _u64(q), _u64(db)
    return np.bitwise_count(qa[:, None, :] ^ da[None, :, :]).sum(-1, dtype=np.int64)


def pack(d, i):
    """(dist, index) -> int64 keys dist << 48 | index, -1 (all ones) where index is -1."""
    d, i = np.asarray(d, np.int64), np.asarray(i, np.int64)
    return np.where(i < 0, np.int64(-1), (d << IDX_BITS) | i)


def unpack(keys):
    """int64 keys (numpy or tensor) -> (dist, index) int64; -1 or NONE -> (-1, -1)."""
    k = keys.cpu().numpy() if isinstance(keys, torch.Tensor) else np.asarray(keys)
    k = k.astype(np.int64)
    none = (k == -1) | (k == NONE)
    d = np.where(none, -1, (k >> IDX_BITS) & 0xFFFF)
    i = np.where(none, -1, k & IDX_MASK)
    return d, i


def _two_smallest(keys):
    """keys (nq, n) int64 -> (nq, 2), ascending, NONE-padded."""
    if keys.shape[1] < 2:
        keys = np.concatenate([keys, np.full((len(keys), 2 - keys.shape[1]), NONE)], 1)
    part = np.partition(keys, 1, axis=1)[:, :2]
    return np.sort(part, axis=1)


def top2_dense(q, db, first_index=0, chunk=4096):
    """Brute force: every (query, row) distance by popcount of the XOR of the 64-bit words."""
    q = np.ascontiguousarray(q, np.uint8).reshape(-1, 32)
    db = np.ascontiguousarray(db, np.uint8).reshape(-1, 32)
    best = np.full((len(q), 2), NONE)
    for lo in range(0, len(db), chunk):
        d = hamming(q, db[lo:lo + chunk])
        rows = np.arange(lo, lo + d.shape[1], dtype=np.int64) + first_index
        best = _two_smallest(np.concatenate([best, (d << IDX_BITS) | rows[None, :]], 1))
    return unpack(best)


def lowest_rows(row_of, npool):
    """(npool, 2) int64: the two lowest rows that hold each pool entry, len(row_of) where there is none.  row_of may be
    a tensor on any device (a 25.6 M-row layout is reduced where it lives)."""
    r = torch.as_tensor(row_of).reshape(-1).long()
    n = r.numel()
    rows = torch.arange(n, device=r.device)
    first = torch.full((npool,), n, dtype=torch.int64, device=r.device).scatter_reduce(0, r, rows, "amin")
    later = rows != first[r]
    second = torch.full((npool,), n, dtype=torch.int64, device=r.device).scatter_reduce(0, r[later], rows[later], "amin")
    return torch.stack([first, second], 1).cpu().numpy()


def top2_pooled(q, pool, row_of, first_index=0):
    """Exact top-2 over db = pool[row_of] at O(nq x |pool| + ndb): rows that hold one pool entry are at one distance
    from every query, so only the two lowest of them can be reported.  The best is the lowest (distance, first row)
    over the pool; the second is the better of the runner-up of that order and the best entry's second row."""
    q = np.ascontiguousarray(q, np.uint8).reshape(-1, 32)
    pool = np.ascontiguousarray(pool, np.uint8).reshape(-1, 32)
    low = lowest_rows(row_of, len(pool))
    n = torch.as_tensor(row_of).numel()
    out = np.empty((len(q), 2), np.int64)
    qchunk = max(1, (1 << 22) // len(pool))
    for lo in range(0, len(q), qchunk):
        d = hamming(q[lo:lo + qchunk], pool)
        k1 = np.where(low[None, :, 0] < n, (d << IDX_BITS) | (low[None, :, 0] + first_index), NONE)
        k2 = np.where(low[None, :, 1] < n, (d << IDX_BITS) | (low[None, :, 1] + first_index), NONE)
        p = np.argmin(k1, axis=1)
        r = np.arange(len(d))
        b = k1[r, p]
        k1[r, p] = NONE
        out[lo:lo + len(d), 0] = b
        out[lo:lo + len(d), 1] = np.minimum(k1.min(1), k2[r, p])
    return unpack(out)


def _signs(bits_u8, dtype):
    """(n, 32) uint8 -> (n, 256) of +1 / -1 (bit 0 / 1); the bit order only has to agree between the two sides."""
    sh = torch.arange(8, device=bits_u8.device, dtype=torch.uint8)
    b = ((bits_u8.unsqueeze(-1) >> sh) & 1).reshape(len(bits_u8), 256)
    return (1 - 2 * b.to(torch.int8)).to(dtype)


def top2_gemm(q, db, first_index=0, chunk=1 << 18):
    """Top-2 through a ±1 matrix product: dot(q, x) = 256 - 2 hamming.  Every partial sum is an integer of magnitude
    <= 256, so the product is exact in float16 (float32 on the CPU) in any reduction order, with TF32 or reduced
    precision allowed.  Per chunk of rows the two smallest hamming << 18 | row keys are kept, then merged."""
    db = torch.as_tensor(db)
    q = torch.as_tensor(q).to(db.device)
    dt = torch.float16 if db.is_cuda else torch.float32
    qs = _signs(q, dt)
    cand = []
    for lo in range(0, len(db), chunk):
        x = _signs(db[lo:lo + chunk], dt)
        dot = (qs @ x.T).to(torch.int32)
        key = (((256 - dot) >> 1) << 18) | torch.arange(len(x), device=db.device, dtype=torch.int32)
        kk = torch.topk(key, min(2, len(x)), dim=1, largest=False).values.long()
        cand.append(((kk >> 18) << IDX_BITS) | ((kk & ((1 << 18) - 1)) + lo + first_index))
        del x, dot, key
    allk = torch.cat(cand, 1).cpu().numpy()
    return unpack(_two_smallest(allk))


def votes(best_keys, th, desc_per_kf, first_kf, n_kf):
    """db_merge_kernel's vote rule, written out: a query votes for the keyframe of this shard that owns its best match
    when best distance <= th (inclusive); rows of other shards, and a missing best, cast nothing.  A short last keyframe
    counts like any other."""
    d, i = unpack(best_keys)
    out = np.zeros(n_kf, np.int64)
    first = first_kf * desc_per_kf
    for dd, ii in zip(d.reshape(-1), i.reshape(-1)):
        if ii < 0 or dd > th:
            continue
        local = ii - first
        if local >= 0 and local // desc_per_kf < n_kf:
            out[local // desc_per_kf] += 1
    return out


Layout = namedtuple("Layout", "kind tile qper tiles qblocks parts tiles_per_cta slice_rows")

KINDS = ("umma", "imma", "popc")


def scan_layout(kind, ndb, nq, n_sm):
    """db_scan's slice arithmetic, line for line (csrc/match.cu, static int db_scan): tile rows, queries per CTA,
    the number of slices and tiles per slice with the 20-bit clamp on the in-slice index."""
    k = {"umma": 0, "imma": 1, "popc": 2}[kind]
    tile = 256 if k == 2 else 128 if k == 1 else 64          # kDbTile / kMmaTile / umma::kTileN
    qper = 128 if k == 2 else 256 if k == 1 else 256         # kDbQPerCta / kMmaQPerCta / umma::kQPerCta
    tiles = (ndb + tile - 1) // tile
    qblocks = (nq + qper - 1) // qper
    parts = max(1, n_sm * (2 if k == 0 else 8) // qblocks)
    parts = min(parts, tiles)
    tpc = (tiles + parts - 1) // parts
    if k != 2:
        tpc = min(tpc, (1 << 20) // tile)
    parts = (tiles + tpc - 1) // tpc
    return Layout(kind, tile, qper, tiles, qblocks, parts, tpc, tpc * tile)


def slice_of(lay, row):
    return row // lay.slice_rows


def slice_starts(lay):
    return [s * lay.slice_rows for s in range(lay.parts)]


def local_tile(lay, row):
    """Tile index inside the row's slice."""
    return (row % lay.slice_rows) // lay.tile


def group(lay, row):
    """db_top2_umma_kernel: the accumulator group (epilogue warps and TMEM stage) that sees the row: local tile % 3."""
    assert lay.kind == "umma"
    return local_tile(lay, row) % 3


def in_tile(lay, row):
    """Position in the tile (the umma accumulator column, the imma B column)."""
    return row % lay.tile


def slice_tiles(lay, s):
    """Number of tiles of slice s (the last one may be short)."""
    return min(lay.tiles_per_cta, lay.tiles - s * lay.tiles_per_cta)
