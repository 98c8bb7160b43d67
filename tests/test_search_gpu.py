"""GPU parity tests proper: CUDA path (through the C ABI) vs the CPU oracle on the same seeded inputs.
Integer/index outputs bit-exact; fp32 scores bit-identical (stricter than the 1e-3 the north star allows)."""
import numpy as np
import pytest

from tests.helpers import assert_topk_equal, load_ivfpq_small, near_queries, opq_matrix, uniform_lens

pytestmark = pytest.mark.gpu
SEED = 1234


def make_pair(oracle, nlist, lens, seed=SEED, explicit=False, shard=None, perm_ids=False):
    from densephrases_b200 import IvfPqIndex
    A = opq_matrix(seed)
    pq = oracle.gen_pq(seed)
    codes = ids = None
    if explicit:
        codes = np.concatenate([oracle.gen_codes(seed + 7, l, 0, int(lens[l])) for l in range(nlist)] + [np.zeros((0, 96), np.uint8)])
        if perm_ids:
            ids = np.random.default_rng(seed).permutation(int(np.sum(lens))).astype(np.int64) * 3 + 11
    ref = oracle.RefIndex(A, pq, lens, centroids=oracle.gen_centroids(seed, 0, nlist), codes=codes, ids=ids, seed=seed)
    gpu = IvfPqIndex(nlist)
    gpu.set_opq(A)
    gpu.gen_pq(seed)
    gpu.gen_centroids(seed)
    if shard is not None:
        gpu.set_shard(*shard)
    if explicit:
        lo, hi = shard if shard is not None else (0, nlist)
        r0, r1 = ref.list_off[lo], ref.list_off[hi - 1] + lens[hi - 1]
        gpu.set_lists(lens, codes[r0:r1], None if ids is None else ids[r0:r1])
    else:
        gpu.set_lists_synthetic(lens, seed)
    return ref, gpu


def test_generators_match_oracle(oracle):
    lens = np.array([40, 0, 33, 1, 64], dtype=np.int64)
    ref, gpu = make_pair(oracle, 5, lens)
    ids = np.arange(ref.ntotal, dtype=np.int64)
    v, f = gpu.reconstruct_batch(ids)
    vr, fr = ref.reconstruct(ids)
    assert f.all() and fr.all()
    assert np.array_equal(v.view(np.int32), vr.view(np.int32))      # centroids + pq + codes + layout all bit-identical
    v2, f2 = gpu.reconstruct_batch(np.array([-1, ref.ntotal, 10**12], dtype=np.int64))
    assert not f2.any() and not v2.any()                              # missing label -> zeros (index.py:287-288)
    assert np.array_equal(gpu.opq_matrix(), ref.A)


@pytest.mark.parametrize("mode", [1, 3, 2, 4, 0])     # exact | single-query gathers | pair-packed | quad-packed gathers | auto
@pytest.mark.parametrize("nlist,N,nprobe,k,nq", [(16, 5000, 4, 10, 9), (64, 40000, 16, 10, 33), (1, 3000, 256, 10, 5),
                                                  (40, 2000, 256, 100, 7), (8, 100, 8, 200, 3)])
def test_search_matches_oracle(oracle, mode, nlist, N, nprobe, k, nq):
    lens = uniform_lens(N, nlist)
    ref, gpu = make_pair(oracle, nlist, lens)
    gpu.nprobe = nprobe
    gpu.set_scan_mode(mode)
    x = np.concatenate([near_queries(ref, nq - 2, 4321), 0.5 * np.random.default_rng(1).standard_normal((2, 768)).astype(np.float32)])
    D, I = gpu.search(x, k)
    Dr, Ir, keyr = ref.search(x, k, nprobe, return_key=True)
    assert np.array_equal(gpu.last_xr(nq).view(np.int32), ref.rotate(x).view(np.int32))
    assert np.array_equal(gpu.last_probes(nq), keyr.astype(np.int32))
    assert_topk_equal(D, I, Dr, Ir, f"mode={mode}")


@pytest.mark.parametrize("mode", [1, 3, 2, 4])
def test_ragged_empty_lists_and_explicit_ids(oracle, mode):
    rng = np.random.default_rng(5)
    nlist = 48
    lens = rng.integers(0, 700, nlist).astype(np.int64)
    lens[[0, 7, 47]] = 0
    lens[3] = 1
    lens[4] = 32
    lens[5] = 33
    ref, gpu = make_pair(oracle, nlist, lens, explicit=True, perm_ids=True)
    gpu.nprobe = 12
    gpu.set_scan_mode(mode)
    x = near_queries(ref, 17, 99)
    D, I = gpu.search(x, 10)
    Dr, Ir = ref.search(x, 10, 12)
    assert_topk_equal(D, I, Dr, Ir)
    v, f = gpu.reconstruct_batch(Ir[0])
    vr, fr = ref.reconstruct(Ir[0])
    assert np.array_equal(v.view(np.int32), vr.view(np.int32)) and f.all()
    # search score == <xr, reconstruct(id)> identity (SURVEY Appendix A)
    xr = ref.rotate(x)
    assert np.abs(v @ xr[0] - D[0]).max() < 1e-3


def test_duplicate_codes_ties(oracle):
    """Identical codes => exactly equal scores (duplicate Wikipedia text, SURVEY 7): canonical tie order."""
    nlist = 4
    lens = np.array([50000, 60000, 70000, 80000], dtype=np.int64)
    from densephrases_b200 import IvfPqIndex
    A = opq_matrix(3)
    pq = oracle.gen_pq(3)
    Cm = oracle.gen_centroids(3, 0, nlist)
    base = oracle.gen_codes(3, 0, 0, 8)
    codes = base[np.random.default_rng(0).integers(0, 8, int(lens.sum()))]      # only 8 distinct code rows
    ref = oracle.RefIndex(A, pq, lens, centroids=Cm, codes=codes)
    for mode in (1, 3, 2, 4):
        gpu = IvfPqIndex(nlist)
        gpu.set_opq(A); gpu.set_pq(pq); gpu.set_centroids(Cm); gpu.set_lists(lens, codes)
        gpu.nprobe = 4
        gpu.set_scan_mode(mode)
        x = near_queries(ref, 6, 1)
        D, I = gpu.search(x, 20)
        Dr, Ir = ref.search(x, 20, 4)
        assert_topk_equal(D, I, Dr, Ir, f"ties mode={mode}")
        # canonical order inside a tie group: scan order (probe rank, offset) ascending == label ascending within a list
        if mode != 1:
            flags = gpu.last_flags(6)
            assert flags.any(), "heavy ties must trip the exactness proof and take the exact fallback"


def test_device_tensor_api_and_fast_equals_exact(oracle):
    import torch
    lens = uniform_lens(200000, 128)
    ref, gpu = make_pair(oracle, 128, lens)
    gpu.nprobe = 32
    x = near_queries(ref, 64, 7)
    xt = torch.from_numpy(x).cuda()
    gpu.set_scan_mode(1)
    D1, I1 = gpu.search(xt, 10)
    for mode in (3, 2, 4, 0):
        gpu.set_scan_mode(mode)
        D0, I0 = gpu.search(xt, 10)
        flags = gpu.last_flags(64)
        assert torch.equal(D0, D1) and torch.equal(I0, I1), f"mode {mode}"
        assert flags.sum() == 0, f"mode {mode}: the filter should prove exactness on generic data"
        assert gpu.last_group_size() == {3: 1, 2: 2, 4: 4, 0: 1}[mode]   # auto: lists of 1562 vectors are too short to amortise the packed-LUT rebuild
    Dr, Ir = ref.search(x, 10, 32)
    assert_topk_equal(D0.cpu().numpy(), I0.cpu().numpy(), Dr, Ir)


def test_golden_fixture_on_gpu(oracle):
    from densephrases_b200 import IvfPqIndex
    g, meta = load_ivfpq_small(oracle)
    for mode in (3, 2, 1):
        ix = IvfPqIndex(len(g["list_len"]))
        ix.set_opq(g["A"]); ix.set_pq(g["pq"]); ix.set_centroids(g["centroids"]); ix.set_lists(g["list_len"], g["codes"], g["ids"])
        ix.nprobe = meta["nprobe"]
        ix.set_scan_mode(mode)
        D, I = ix.search(g["x"], meta["k"])
        assert np.array_equal(ix.last_probes(len(g["x"])), g["key"].astype(np.int32))
        assert_topk_equal(D, I, g["D"], g["I"], f"golden mode={mode}")
        assert np.array_equal(ix.reconstruct_batch(g["I"][0])[0].view(np.int32), g["recon0"].view(np.int32))


@pytest.mark.parametrize("nshards", [2, 5, 3])
def test_list_range_shards_on_one_device(oracle, nshards):
    """The multi-GPU data path (per-shard partial top-k + merge_shards) exercised with all shards on cuda:0."""
    import torch
    from densephrases_b200 import IvfPqIndex, merge_shards
    from densephrases_b200.sharded import shard_ranges
    rng = np.random.default_rng(8)
    nlist = 96
    lens = (np.exp(rng.normal(0, 0.5, nlist)) * 1500).astype(np.int64)     # log-normal skew (SURVEY 8d)
    lens[5] = 0
    ref, _ = make_pair(oracle, nlist, lens)
    x = near_queries(ref, 40, 12)
    xt = torch.from_numpy(x).cuda()
    k, nprobe = 10, 24
    shards = []
    for si, (lo, hi) in enumerate(shard_ranges(lens, nshards)):
        _, sh = make_pair(oracle, nlist, lens, shard=(lo, hi))
        sh.nprobe = nprobe
        sh.set_scan_mode((2, 3, 4)[si % 3])                  # mix pair-packed, single-query and quad-packed shards
        assert sh.ntotal_local == int(lens[lo:hi].sum()) and sh.ntotal == int(lens.sum())
        shards.append(sh)
    if nshards == 2:      # replicated coarse quantizer: every shard selects the global probes itself
        parts = [sh.search_partial(xt, k) for sh in shards]
    elif nshards == 3:    # query-split coarse quantizer: shard r assigns ITS SLICE of the batch over all lists -> "all-gather" of records
        per = (len(x) + nshards - 1) // nshards
        rec = torch.cat([sh.coarse_split(xt[r * per:(r + 1) * per].contiguous()) for r, sh in enumerate(shards)]).contiguous()
        assert rec.shape == (len(x), 768 + 2 * nprobe)
        parts = [sh.search_assigned(rec, k) for sh in shards]
        keyr = ref.search(x, k, nprobe, return_key=True)[2].astype(np.int32)
        assert np.array_equal(shards[0].last_probes(len(x)), keyr) and np.array_equal(shards[2].last_probes(len(x)), keyr)
        assert np.array_equal(shards[1].last_xr(len(x)).view(np.int32), ref.rotate(x).view(np.int32))
    else:                 # sharded coarse quantizer: per-shard candidates -> "all-gather" -> merge -> preassigned search
        keys_g = torch.stack([sh.coarse_local(xt) for sh in shards]).contiguous()
        parts = [sh.search_preassigned(keys_g, k) for sh in shards]
        assert np.array_equal(shards[0].last_probes(len(x)), ref.search(x, k, nprobe, return_key=True)[2].astype(np.int32))
    Dg, Ig, Gg = (torch.stack([p[i] for p in parts]).contiguous() for i in range(3))
    D, I = merge_shards(Dg, Ig, Gg, k)
    from densephrases_b200.ivfpq import merge_shards_packed, pack_topk
    D2, I2 = merge_shards_packed(torch.stack([pack_topk(*p) for p in parts]).contiguous(), k)      # the single-buffer exchange
    assert torch.equal(D, D2) and torch.equal(I, I2)
    Dr, Ir = ref.search(x, k, nprobe)
    assert_topk_equal(D.cpu().numpy(), I.cpu().numpy(), Dr, Ir, "sharded")
    # a label that lives in another shard reconstructs to zeros + found=0 on this shard; the sum over shards is the vector
    lo, hi = shard_ranges(lens, nshards)[0]
    _, sh0 = make_pair(oracle, nlist, lens, shard=(lo, hi))
    v, f = sh0.reconstruct_batch(Ir[0])
    l, _ = ref.locate(Ir[0])
    assert np.array_equal(f.astype(bool), (l >= lo) & (l < hi))
    assert not v[~f.astype(bool)].any()


def test_mid_size_skewed_lists_and_large_k(oracle):
    rng = np.random.default_rng(3)
    nlist = 512
    lens = (np.exp(rng.normal(0, 0.5, nlist)))
    lens = (lens / lens.sum() * 5_000_000).astype(np.int64)
    ref, gpu = make_pair(oracle, nlist, lens)
    gpu.nprobe = 64
    x = near_queries(ref, 32, 5)
    for k, mode in ((10, 2), (10, 3), (10, 4), (60, 4), (400, 2), (400, 4), (400, 0), (1024, 0)):   # top_k up to 200 x2 in the reference (Makefile:490, model.py:79-81)
        gpu.set_scan_mode(mode)
        D, I = gpu.search(x, k)
        Dr, Ir = ref.search(x, k, 64)
        assert_topk_equal(D, I, Dr, Ir, f"k={k} mode={mode}")
        assert gpu.last_flags(32).sum() <= (1 if mode == 4 else 0)       # quad filter (8-bit LUTs): a rare proof failure only costs an exact re-run


def test_coarse_ties_duplicate_centroids(oracle):
    """Exactly equal coarse scores (duplicated centroids) at the nprobe boundary: the smaller list id is probed (an equal score
    never evicts in faiss' heap either); probe SETS and final results must match the oracle."""
    from densephrases_b200 import IvfPqIndex
    nlist, nprobe = 96, 12
    lens = np.full(nlist, 200, dtype=np.int64)
    A, pq = opq_matrix(2), oracle.gen_pq(2)
    Cm = oracle.gen_centroids(2, 0, nlist)
    Cm[1::2] = Cm[0::2]                                  # every centroid appears twice
    codes = np.concatenate([oracle.gen_codes(2, l, 0, 200) for l in range(nlist)])
    ref = oracle.RefIndex(A, pq, lens, centroids=Cm, codes=codes)
    x = near_queries(ref, 20, 3)
    Dr, Ir, keyr = ref.search(x, 10, nprobe, return_key=True)
    for mode in (3, 2):
        gpu = IvfPqIndex.from_arrays(A, Cm, pq, lens, codes)
        gpu.nprobe = nprobe
        gpu.set_scan_mode(mode)
        D, I = gpu.search(x, 10)
        pr = gpu.last_probes(20)
        assert all(set(pr[i].tolist()) == set(keyr[i].tolist()) for i in range(20))
        assert_topk_equal(D, I, Dr, Ir, f"coarse ties mode={mode}")


def test_large_nlist_uses_generic_coarse_select(oracle):
    """nlist above the shared-memory fast path (16384) takes the generic radix-select kernel; both must agree with the oracle."""
    nlist = 20000
    lens = np.full(nlist, 3, dtype=np.int64)
    ref, gpu = make_pair(oracle, nlist, lens)
    gpu.nprobe = 40
    x = near_queries(ref, 6, 8)
    D, I = gpu.search(x, 10)
    Dr, Ir, keyr = ref.search(x, 10, 40, return_key=True)
    assert np.array_equal(gpu.last_probes(6), keyr.astype(np.int32))
    assert_topk_equal(D, I, Dr, Ir)


@pytest.mark.parametrize("nprobe", [24, 300])
def test_long_rows_chunked_select_both_coarse_paths(oracle, nprobe):
    """Rows longer than the shared-memory select (nlist > 16384) are selected chunk by chunk (8192 lists per CTA) and merged per query:
    the tensor-core candidate keys and the exact SIMT scores both go through it and must reproduce the oracle's probes and scores."""
    nlist = 20000
    lens = np.full(nlist, 2, dtype=np.int64)
    ref, gpu = make_pair(oracle, nlist, lens)
    gpu.nprobe = nprobe
    x = np.concatenate([near_queries(ref, 30, 5), 0.5 * np.random.default_rng(3).standard_normal((10, 768)).astype(np.float32)])
    Dr, Ir, keyr = ref.search(x, 10, nprobe, return_key=True)
    cdr, _ = ref.coarse(ref.rotate(x), nprobe)
    for tc in (1, 0):
        gpu.set_coarse_tc(tc)
        D, I = gpu.search(x, 10)
        pr = gpu.last_probes(len(x))
        # exact score ties between two lists do occur at this size: the CUDA order is canonical (score desc, list asc), faiss' / the
        # oracle's is heap-dependent -> compare the probe SETS and the (sorted) scores bit for bit
        assert all(set(pr[i].tolist()) == set(keyr[i].tolist()) for i in range(len(x))), f"probes differ (tc={tc})"
        assert np.array_equal(gpu.last_coarse(len(x)).view(np.int32), cdr.view(np.int32)), f"coarse scores differ (tc={tc})"
        if tc == 1:
            pr_tc = pr.copy()
        else:
            assert np.array_equal(pr, pr_tc), "tensor-core and SIMT coarse paths order the probes differently"
        assert_topk_equal(D, I, Dr, Ir, f"tc={tc}")


@pytest.mark.parametrize("nprobe", [8, 256])
def test_tensor_core_coarse_is_bit_identical(oracle, nprobe):
    """Coarse quantizer on tcgen05 (3xTF32 candidates + exact re-rank + proof) == SIMT sequential-k path == oracle (probes AND scores)."""
    nlist = 1024
    lens = np.full(nlist, 40, dtype=np.int64)
    ref, gpu = make_pair(oracle, nlist, lens)
    gpu.nprobe = nprobe
    x = np.concatenate([near_queries(ref, 60, 5), 0.5 * np.random.default_rng(2).standard_normal((36, 768)).astype(np.float32)])
    out = {}
    for tc in (1, 0):
        gpu.set_coarse_tc(tc)
        D, I = gpu.search(x, 10)
        out[tc] = (gpu.last_probes(len(x)).copy(), gpu.last_coarse(len(x)).copy(), D, I)
    Dr, Ir, keyr = ref.search(x, 10, nprobe, return_key=True)
    cdr, _ = ref.coarse(ref.rotate(x), nprobe)
    for tc in (1, 0):
        assert np.array_equal(out[tc][0], keyr.astype(np.int32)), f"probes differ (tc={tc})"
        assert np.array_equal(out[tc][1].view(np.int32), cdr.view(np.int32)), f"coarse scores differ (tc={tc})"
        assert_topk_equal(out[tc][2], out[tc][3], Dr, Ir, f"tc={tc}")


def test_tensor_core_coarse_repair_path(oracle):
    """Near-identical centroids: candidate scores sit inside the error bound, the proof fails, and every query takes the repair path
    (exact scores for all lists) -- results must still equal the oracle."""
    from densephrases_b200 import IvfPqIndex
    nlist, nprobe = 256, 16
    rng = np.random.default_rng(4)
    lens = np.full(nlist, 30, dtype=np.int64)
    A, pq = opq_matrix(4), oracle.gen_pq(4)
    Cm = (oracle.gen_centroids(4, 0, 1) + 1e-6 * rng.standard_normal((nlist, 768))).astype(np.float32)
    codes = np.concatenate([oracle.gen_codes(4, l, 0, 30) for l in range(nlist)])
    ref = oracle.RefIndex(A, pq, lens, centroids=Cm, codes=codes)
    gpu = IvfPqIndex.from_arrays(A, Cm, pq, lens, codes)
    gpu.nprobe = nprobe
    x = near_queries(ref, 48, 6)
    out = {}
    for tc in (1, 0):        # both paths are canonical (score desc, list asc): they must agree exactly, ties included
        gpu.set_coarse_tc(tc)
        D, I = gpu.search(x, 10)
        out[tc] = (gpu.last_probes(48).copy(), gpu.last_coarse(48).copy(), D, I)
    assert np.array_equal(out[1][0], out[0][0]) and np.array_equal(out[1][1].view(np.int32), out[0][1].view(np.int32))
    assert np.array_equal(out[1][2].view(np.int32), out[0][2].view(np.int32)) and np.array_equal(out[1][3], out[0][3])
    cdr, _ = ref.coarse(ref.rotate(x), nprobe)
    assert np.array_equal(out[1][1].view(np.int32), cdr.view(np.int32))     # the exact coarse scores equal the oracle's bit for bit


def test_quad_mode_is_the_default_for_shared_long_lists(oracle):
    """Lists of >= 4096 vectors probed by several queries of the batch -> four queries share every gather (scan_quad_kernel);
    groups of 1, 2, 3 and 4 queries per list all occur (33 queries x 6 probes over 12 lists), k + slack stays within the buffers."""
    lens = uniform_lens(12 * 4500, 12)
    ref, gpu = make_pair(oracle, 12, lens)
    gpu.nprobe = 6
    x = near_queries(ref, 33, 21)
    for k in (10, 40):
        D, I = gpu.search(x, k)
        assert gpu.last_group_size() == 4
        Dr, Ir = ref.search(x, k, 6)
        assert_topk_equal(D, I, Dr, Ir, f"quad k={k}")
    D, I = gpu.search(x, 300)                  # k + slack no longer fits the quad buffers -> pair-packed
    assert gpu.last_group_size() == 2
    assert_topk_equal(D, I, *ref.search(x, 300, 6), "pair fallback")


def test_merge_shards_many_candidates():
    """nshards * k in (4096, 8192] needs the opted-in 64 KB of dynamic shared memory (8 shards x k = 1024)."""
    import torch
    from densephrases_b200 import merge_shards
    g = torch.Generator().manual_seed(0)
    nsh, n, k = 8, 3, 1024
    Dg = torch.randn((nsh, n, k), generator=g).sort(dim=2, descending=True).values.cuda().contiguous()
    Gg = torch.randperm(nsh * n * k, generator=g).to(torch.int32).view(nsh, n, k).cuda().contiguous()
    Ig = (Gg.to(torch.int64) + 7).contiguous()
    D, I = merge_shards(Dg, Ig, Gg, k)
    flat = Dg.permute(1, 0, 2).reshape(n, -1)
    top = flat.sort(dim=1, descending=True).values[:, :k]
    assert torch.equal(D, top)


def test_chunked_upload_and_device_built_direct_map(oracle, monkeypatch):
    """set_lists streams the list-major rows through a bounded staging buffer (here forced to 700 rows per chunk, lists of up to
    2000 rows) and builds the label -> row direct map on the device (thrust sort): search, explicit labels and reconstruct of
    permuted labels all equal the oracle."""
    from densephrases_b200 import IvfPqIndex
    monkeypatch.setenv("DPH_UPLOAD_CHUNK_ROWS", "700")
    rng = np.random.default_rng(11)
    nlist = 40
    lens = rng.integers(0, 2000, nlist).astype(np.int64)
    lens[3] = 0
    N = int(lens.sum())
    codes = rng.integers(0, 256, (N, 96), dtype=np.uint8)
    ids = rng.permutation(N).astype(np.int64) * 3 + 1                 # sparse, shuffled labels
    A, pq, Cm = opq_matrix(2), oracle.gen_pq(2), oracle.gen_centroids(2, 0, nlist)
    ref = oracle.RefIndex(A, pq, lens, centroids=Cm, codes=codes, ids=ids)
    gpu = IvfPqIndex.from_arrays(A, Cm, pq, lens, codes, ids)
    gpu.nprobe = 12
    x = near_queries(ref, 17, 4)
    D, I = gpu.search(x, 10)
    assert_topk_equal(D, I, *ref.search(x, 10, 12), "chunked upload")
    probe = np.concatenate([ids[rng.integers(0, N, 50)], [0, 2, -5, 3 * N + 7]])       # labels that do not exist -> zeros, found 0
    v, f = gpu.reconstruct_batch(probe)
    vr, fr = ref.reconstruct(probe)
    assert np.array_equal(f, fr) and np.array_equal(v.view(np.int32), vr.view(np.int32))
