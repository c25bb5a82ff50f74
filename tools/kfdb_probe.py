"""KeyFrameDatabase queries on the GPU (swarmmap_b200.kfdb) against the CPU oracle on one host core; prints one JSON line.

Keyframes: BowVectors of frames from synth.make_sequence, extracted by the GPU extractor (1000 features, 8 levels)
and transformed with a k=10, L=5 synthetic vocabulary (levelsup 4, as Frame::ComputeBoW).  A database of n keyframes
cycles through the extracted frames; every copy after the first drops a random 10 % of its words, so no two keyframes
are the same.  GetBestCovisibilityKeyFrames(10) of keyframe i: the 10 nearest sequence indices.  Queries: later
frames (not in the database) and noisy re-renders of database keyframes (planted revisits), half each.

For each database size (1 k, 10 k, 50 k) and batch size (1, 128), in both modes: queries/s from the device events
around query + finish, and end to end (host clock around the synchronised two-phase call); the oracle's queries/s at
the same sizes; and, on a fresh database pair, the parity of 128 sampled queries (ordered scored lists, float score
bits, ordered candidates) against the oracle."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from swarmmap_b200 import synth  # noqa: E402


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def frames_bows(n_frames, vocab):
    from swarmmap_b200.orb import ORBextractor
    ex = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=64)
    seq = synth.make_sequence(n_frames, seed=20261020)
    out = []
    for b in range(0, n_frames, 64):
        imgs = np.stack(seq[b:b + 64])
        _, desc, n = ex.extract_batch(imgs)
        out += vocab.transform_batch(desc, n, 4)
    return [(r.word_ids, r.values) for r in out]


def perturb(rng, bow, drop=0.1):
    w, v = bow
    keep = rng.random(len(w)) >= drop
    return w[keep], v[keep] / max(v[keep].sum(), 1e-300)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000,10000,50000")
    ap.add_argument("--batches", default="1,128")
    ap.add_argument("--frames", type=int, default=1200)
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()
    import oracle_kfdb_lib as okl
    from swarmmap_b200.bow import ORBVocabulary
    from swarmmap_b200.kfdb import KeyFrameDatabase
    sizes = [int(x) for x in args.sizes.split(",")]
    batches = [int(x) for x in args.batches.split(",")]
    vocab = ORBVocabulary(synth.make_vocabulary(10, 5, seed=20261020))
    base = frames_bows(args.frames, vocab)
    n_db_frames = args.frames - 200  # the last 200 frames are never in a database: "later frames" queries
    rng = np.random.default_rng(1)
    res = dict(device=device_info(), vocab_words=vocab.n_words, frames=args.frames,
               mean_words_per_kf=float(np.mean([len(b[0]) for b in base])), results=[], parity=[])
    for n in sizes:
        bows = [base[i % n_db_frames] if i < n_db_frames else perturb(rng, base[i % n_db_frames]) for i in range(n)]
        ids = np.arange(n, dtype=np.uint64) + 1
        nb = {int(i + 1): [int(j + 1) for j in sorted((j for j in range(max(0, i - 5), min(n, i + 6)) if j != i),
                                                       key=lambda j: (abs(j - i), j))][:10] for i in range(n)}
        qs = [base[n_db_frames + k % 200] if k % 2 == 0 else perturb(rng, bows[int(rng.integers(n))], 0.2)
              for k in range(128)]
        ms = np.full(128, 0.01, np.float32)
        conn = [nb.get(int(rng.integers(1, n + 1)), []) for _ in range(128)]
        # parity on a fresh pair
        g, o = KeyFrameDatabase(vocab), okl.KeyFrameDatabase(vocab.n_words)
        g.add(ids, bows)
        for i, b in zip(ids, bows):
            o.add(int(i), b)
        o.set_neighbours(nb)
        for mode in (0, 1):
            cand = g.detect_relocalization_candidates(qs, nb) if mode == 0 else g.detect_loop_candidates(qs, ms, conn, nb)
            ok, n_cand = True, 0
            for q in range(128):
                sid, ssc, cid = o.query(mode, qs[q], ms[q] if mode else 0.0, conn[q] if mode else ())
                gid, gsc = g.last_scored[q]
                ok &= np.array_equal(gid, sid) and np.array_equal(gsc.view(np.uint32), ssc.view(np.uint32))
                ok &= np.array_equal(cand[q], cid)
                n_cand += len(cid)
            res["parity"].append(dict(n_kf=n, mode=["reloc", "loop"][mode], queries=128, identical=bool(ok),
                                      candidates=n_cand))
        # timing (same database, after the parity queries)
        for mode in (0, 1):
            for bsz in batches:
                qb = qs[:bsz]

                def call():
                    if mode == 0:
                        return g.detect_relocalization_candidates(qb, nb)
                    return g.detect_loop_candidates(qb, ms[:bsz], conn[:bsz], nb)
                call()
                call()
                dev, t0 = 0.0, time.perf_counter()
                for _ in range(args.iters):
                    call()
                    dev += g.last_device_ms()
                wall = time.perf_counter() - t0
                t_or = o.time_queries(mode, qb, ms[:bsz], 1)
                res["results"].append(dict(n_kf=n, mode=["reloc", "loop"][mode], batch=bsz,
                                           gpu_device_qps=bsz * args.iters / (dev / 1e3),
                                           gpu_end_to_end_qps=bsz * args.iters / wall,
                                           oracle_1core_qps=bsz / t_or))
        del g, o
    res["parity_all"] = all(p["identical"] for p in res["parity"])
    print(json.dumps(res))


if __name__ == "__main__":
    main()
