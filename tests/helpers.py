"""Shared test helpers: matched (oracle, CUDA) index pairs and the top-k comparator."""
import numpy as np

D_MODEL = 768


def opq_matrix(seed, d=D_MODEL):
    rng = np.random.default_rng(seed)
    return np.linalg.qr(rng.standard_normal((d, d)))[0].astype(np.float32)


def uniform_lens(N, nlist):
    base, rem = divmod(N, nlist)
    return np.array([base + (1 if l < rem else 0) for l in range(nlist)], dtype=np.int64)


def near_queries(ref, n, seed, noise=0.3):
    """SURVEY 8d 'near' queries: q = A^T (centroid + decode(code_j)) + N(0, noise^2)."""
    rng = np.random.default_rng(seed)
    ids = rng.integers(0, max(ref.ntotal, 1), n)
    v, _ = ref.reconstruct(ids) if ref.ids is None else ref.reconstruct(ref.ids[ids])
    q = v @ ref.A            # un-rotate: A^T v  (row-vector form v A)
    return (q + noise * rng.standard_normal(q.shape)).astype(np.float32)


def ivfpq_small_arrays(oracle, meta, list_len):
    """The seeded part of the tests/golden/ivfpq_small index: matrix, PQ codebooks, centroids and codes from the oracle's generators."""
    seed, nlist = meta["seed"], len(list_len)
    return {"A": oracle.gen_centroids(meta["opq_seed"], 0, D_MODEL, D_MODEL, meta["opq_sigma"]), "pq": oracle.gen_pq(seed),
            "centroids": oracle.gen_centroids(seed, 0, nlist),
            "codes": np.concatenate([oracle.gen_codes(seed, l, 0, int(list_len[l])) for l in range(nlist)])}


def load_ivfpq_small(oracle):
    """tests/golden/ivfpq_small.{npz,json} (tests/golden/make_golden.py) as (arrays, meta), the seeded arrays regenerated."""
    import json
    import os
    gd = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    meta = json.load(open(os.path.join(gd, "ivfpq_small.json")))
    g = dict(np.load(os.path.join(gd, "ivfpq_small.npz")))
    g.update(ivfpq_small_arrays(oracle, meta, g["list_len"]))
    return g, meta


def jsonable(obj):
    """`obj` as it reads back from a JSON golden file: tuples become lists, numpy scalars and arrays Python values."""
    import json

    def numpy_value(o):
        if isinstance(o, (np.ndarray, np.generic)):
            return o.tolist()
        raise TypeError(f"not JSON serializable: {type(o).__name__}")
    return json.loads(json.dumps(obj, default=numpy_value))


def assert_topk_equal(D, I, Dref, Iref, what=""):
    """Bit-identical scores; identical labels up to permutations inside exactly-equal-score groups (faiss' heap
    order among equal scores is unspecified); in the boundary group only the group size is compared."""
    D = np.asarray(D); I = np.asarray(I); Dref = np.asarray(Dref); Iref = np.asarray(Iref)
    assert D.shape == Dref.shape and I.shape == Iref.shape, what
    bits, bits_ref = D.view(np.int32), Dref.view(np.int32)
    bad = np.argwhere(bits != bits_ref)
    assert bad.size == 0, f"{what}: score bits differ at {bad[:5].tolist()}: {D[tuple(bad[0])]!r} vs {Dref[tuple(bad[0])]!r}"
    for r in range(D.shape[0]):
        if np.array_equal(I[r], Iref[r]):
            continue
        last = D[r, -1]
        for v in np.unique(D[r]):
            a, b = sorted(I[r][D[r] == v].tolist()), sorted(Iref[r][Dref[r] == v].tolist())
            if v == last:
                assert len(a) == len(b), f"{what}: row {r} boundary tie group size"
            else:
                assert a == b, f"{what}: row {r} labels differ at score {v}: {a} vs {b}"
