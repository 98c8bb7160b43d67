"""CPU tests of the oracle itself (the reference holds no golden vectors for this path, SURVEY.md 8c):
C restatement == numpy restatement bit-for-bit, both == exhaustive fp64 scoring, heap/tie/padding semantics,
and the committed golden fixtures (tests/golden/make_golden.py) still reproduce."""
import numpy as np
import pytest

from tests.helpers import load_ivfpq_small, near_queries, opq_matrix, uniform_lens


def small_index(oracle, nlist=16, seed=11, lens=None, explicit=False):
    rng = np.random.default_rng(seed)
    if lens is None:
        lens = rng.integers(0, 200, nlist).astype(np.int64)
        lens[3] = 0
    A = opq_matrix(seed)
    pq = oracle.gen_pq(seed)
    Cm = oracle.gen_centroids(seed, 0, nlist)
    codes = None
    if explicit:
        codes = np.concatenate([oracle.gen_codes(seed, l, 0, int(lens[l])) for l in range(nlist)])
    return oracle.RefIndex(A, pq, lens, centroids=Cm, codes=codes, seed=seed)


def test_fma32_emulation_is_exact(oracle):
    rng = np.random.default_rng(0)
    a, b, c = (rng.standard_normal(200000).astype(np.float32) * s for s in (1.0, 3.0, 0.5))
    ref = (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64))      # one rounding to fp64 of the exact value...
    got = oracle.fma32(a, b, c)
    # the exact a*b+c needs <= 24+24+... bits; compare against python's exact rational arithmetic on a sample
    from fractions import Fraction
    for i in rng.integers(0, len(a), 300):
        exact = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        cand = np.float32(float(exact))            # float(Fraction) is correctly rounded to fp64; fp64->fp32 may double round
        lo, hi = np.nextafter(cand, np.float32(-np.inf)), np.nextafter(cand, np.float32(np.inf))
        best = min((lo, cand, hi), key=lambda v: abs(Fraction(float(v)) - exact))
        assert got[i] == best
    assert np.abs(got - ref.astype(np.float32)).max() <= np.spacing(np.abs(ref).astype(np.float32)).max()


def test_c_equals_numpy_restatement(oracle):
    ix = small_index(oracle)
    x = np.random.default_rng(1).standard_normal((5, 768)).astype(np.float32) * 0.5
    D, I, key = ix.search(x, 10, 4, return_key=True)
    D2, I2, key2 = oracle.np_search(ix, x, 10, 4)
    assert np.array_equal(key, key2)
    assert np.array_equal(D.view(np.int32), D2.view(np.int32))
    assert np.array_equal(I, I2)
    assert np.array_equal(ix.rotate(x).view(np.int32), oracle.np_rotate(x, ix.A).view(np.int32))


def test_matches_fp64_brute_force(oracle):
    ix = small_index(oracle, nlist=32, seed=5)
    x = near_queries(ix, 8, 3)
    D, I, key = ix.search(x, 10, 8, return_key=True)
    Db, Ib = oracle.brute_force_fp64(ix, x, key, 10)
    assert np.abs(Db - D).max() < 1e-3          # fp32 sequential-FMA chain vs fp64 (the north-star tolerance)
    assert (Ib == I).mean() > 0.98              # near-ties at 1e-5 may swap neighbours
    for r in range(len(x)):
        assert set(Ib[r]) == set(I[r]) or np.abs(np.sort(Db[r]) - np.sort(D[r].astype(np.float64))).max() < 1e-3


def test_score_is_dot_with_reconstruction(oracle):
    ix = small_index(oracle, explicit=True)
    x = near_queries(ix, 4, 9)
    D, I = ix.search(x, 5, 6)
    xr = ix.rotate(x)
    for r in range(4):
        v, found = ix.reconstruct(I[r])
        assert found.all()
        assert np.abs(v.astype(np.float64) @ xr[r].astype(np.float64) - D[r]).max() < 1e-3


def test_nlist_smaller_than_nprobe_and_padding(oracle):
    """C1-style IVF1 with nprobe 256 (slots beyond nlist are -1) and k larger than the index (faiss pads (-FLT_MAX,-1))."""
    ix = small_index(oracle, nlist=1, lens=np.array([7], dtype=np.int64))
    x = near_queries(ix, 3, 2)
    D, I, key = ix.search(x, 10, 256, return_key=True)
    assert (key[:, 0] == 0).all() and (key[:, 1:] == -1).all()
    assert (I[:, 7:] == -1).all() and (D[:, 7:] == np.float32(-3.4028234663852886e38)).all()
    assert (np.diff(D[:, :7], axis=1) <= 0).all() and (np.sort(I[:, :7], axis=1) == np.arange(7)).all()


def test_missing_labels_reconstruct_to_zero(oracle):
    ix = small_index(oracle)
    v, found = ix.reconstruct(np.array([-1, ix.ntotal, 0], dtype=np.int64))
    assert found.tolist() == [0, 0, 1] and not v[:2].any() and v[2].any()


def test_strict_heap_keeps_earlier_on_ties(oracle):
    """faiss: `if (simi[0] < dis)` -- an equal score never evicts (SURVEY Appendix A)."""
    lens = np.array([6], dtype=np.int64)
    A = np.eye(768, dtype=np.float32)
    pq = np.zeros((96, 256, 8), dtype=np.float32)
    ix = oracle.RefIndex(A, pq, lens, centroids=np.ones((1, 768), np.float32), codes=np.zeros((6, 96), np.uint8))
    D, I = ix.search(np.ones((1, 768), np.float32), 3, 1)
    assert (D == 768.0).all() and sorted(I[0].tolist()) == [0, 1, 2]


def test_resident_lists_view_is_equivalent(oracle):
    ix = small_index(oracle, nlist=64, seed=21, lens=uniform_lens(20000, 64))
    x = near_queries(ix, 4, 2)
    D, I, key = ix.search(x, 10, 8, return_key=True)
    D2, I2 = ix.with_resident_lists(key).search(x, 10, 8)
    assert np.array_equal(D, D2) and np.array_equal(I, I2)


def test_golden_fixture_reproduces(oracle):
    g, meta = load_ivfpq_small(oracle)
    ix = oracle.RefIndex(g["A"], g["pq"], g["list_len"], centroids=g["centroids"], codes=g["codes"], ids=g["ids"])
    D, I, key = ix.search(g["x"], meta["k"], meta["nprobe"], return_key=True)
    assert np.array_equal(D.view(np.int32), g["D"].view(np.int32)) and np.array_equal(I, g["I"]) and np.array_equal(key, g["key"])
    assert np.array_equal(ix.reconstruct(g["I"][0])[0].view(np.int32), g["recon0"].view(np.int32))
