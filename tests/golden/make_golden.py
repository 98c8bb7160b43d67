"""Generates tests/golden/ivfpq_small.{npz,json}: a small explicit IVF-PQ index (permuted labels, ragged and empty
lists), queries, and the oracle's outputs (C restatement, cross-checked against the numpy restatement and the fp64
brute force before writing).  The reference repo has no golden vectors for this path (SURVEY.md 8c) and faiss cannot be
installed here, so these pin the *restatement* (and through it the CUDA path) against silent drift.
The matrix, codebooks, centroids and codes come from the oracle's seeded integer-hash generators, which give the same bits on
every platform, so only labels, queries and outputs are stored (tests.helpers.load_ivfpq_small rebuilds the rest).
Run from the repo root:  python tests/golden/make_golden.py"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ivfpq_ref as R  # noqa: E402
from tests.helpers import ivfpq_small_arrays  # noqa: E402

if __name__ == "__main__":
    R.build()
    # opq_seed / opq_sigma: a dense seeded matrix stands in for the OPQ rotation (the search does not assume orthogonality)
    meta = {"seed": 777, "opq_seed": 778, "opq_sigma": 0.036, "k": 10, "nprobe": 6, "generator": "tests/golden/make_golden.py",
            "oracle": "oracle/ivfpq_ref.c"}
    seed, nlist, k, nprobe = meta["seed"], 24, meta["k"], meta["nprobe"]
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 90, nlist).astype(np.int64)
    lens[[2, 23]] = 0
    lens[5] = 33
    g = ivfpq_small_arrays(R, meta, lens)
    A = g["A"]
    ids = (rng.permutation(int(lens.sum())) * 5 + 3).astype(np.int64)
    ix = R.RefIndex(A, g["pq"], lens, centroids=g["centroids"], codes=g["codes"], ids=ids)
    pick = rng.integers(0, len(ids), 12)
    x = (ix.reconstruct(ids[pick])[0] @ A + 0.3 * rng.standard_normal((12, 768))).astype(np.float32)
    D, I, key = ix.search(x, k, nprobe, return_key=True)
    D2, I2, key2 = R.np_search(ix, x, k, nprobe)
    assert np.array_equal(D.view(np.int32), D2.view(np.int32)) and np.array_equal(I, I2) and np.array_equal(key, key2)
    Db, Ib = R.brute_force_fp64(ix, x, key, k)
    assert np.abs(Db - D).max() < 1e-3 and (Ib == I).mean() > 0.97   # 1e-3 = the north-star score tolerance
    out = os.path.dirname(os.path.abspath(__file__))
    np.savez_compressed(os.path.join(out, "ivfpq_small.npz"), list_len=lens, ids=ids, x=x, D=D, I=I, key=key, recon0=ix.reconstruct(I[0])[0])
    json.dump(meta, open(os.path.join(out, "ivfpq_small.json"), "w"))
    print("wrote", out)
