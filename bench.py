#!/usr/bin/env python
"""bench.py -- queries/sec top-10 over the synthetic PQ96 phrase index (BASELINE.json metric), one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # this repo's CUDA path
  python bench.py --impl reference [...]                          # the reference's CPU path (FAISS-equivalent restatement)

A *step* is one pass of the hot path (OPQ rotation -> coarse top-nprobe -> LUT -> PQ96 scan -> top-k merge) over one
batch of synthetic d=768 vector queries (SURVEY.md 8d: seed 1234 index, seed 4321 "near" queries), k = 10.

  N = 1   C2 (BASELINE.json configs[1]): 100M phrases, IVF4096,PQ96, batch 64, nprobe 256 (the reference's fixed value,
          densephrases/index.py:53,62).  Extra legs in the same line: C1 (configs[0]), the encoder + C3 (configs[2]), and C4's
          1B-phrase index held by this ONE GPU (96 GB) so that the metric's "@1/2/4/8 B200" series has its N=1 point.
  N >= 2  C4 (configs[3]): 1B phrases, IVF65536,PQ96, batch 1024, list-range shards over the N ranks (strong scaling: the
          index and the batch are fixed), `value` at the reference's nprobe 256; the `nprobe32` object holds the same
          measurement at nprobe 32 (BASELINE.md: C4 is reported at nprobe 256 AND 32).
Both arms draw the SAME query vectors (make_query_plan / finish_queries).  Prints ONE JSON line on rank 0.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED_INDEX, SEED_QUERY = 1234, 4321
D, K_TOP, NPROBE = 768, 10, 256
METRIC = "queries/sec top-10 over PQ96 phrase index"


def opq_matrix(seed):
    rng = np.random.default_rng(seed)
    return np.linalg.qr(rng.standard_normal((D, D)))[0].astype(np.float32)


def uniform_lens(N, nlist):
    base, rem = divmod(N, nlist)
    lens = np.full(nlist, base, dtype=np.int64)
    lens[:rem] += 1
    return lens


def workload(name, scale=1.0):
    """BASELINE.json configs by name; `scale` (debug only) shrinks the number of phrases, never the shape."""
    spec = {"C1": (1_000_000, 1, 100), "C2": (100_000_000, 4096, 64), "C4": (1_000_000_000, 65536, 1024)}[name]
    N = max(int(spec[0] * scale), spec[1])
    return dict(name=name, N=N, nlist=spec[1], batch=spec[2], nprobe=NPROBE, k=K_TOP, lens=uniform_lens(N, spec[1]))


def workload_for(n_gpus, scale=1.0):
    return workload("C2" if n_gpus == 1 else "C4", scale)


def config_dict(wl, n_gpus, nprobe=None):
    nprobe = wl["nprobe"] if nprobe is None else nprobe
    per_gpu_gb = wl["N"] * 96 / n_gpus / 1e9
    return {"workload": f"{wl['name']}: {wl['N']}-phrase IVF{wl['nlist']},PQ96 (OPQ96) index, batch {wl['batch']} d=768 near queries, "
                        f"nprobe {nprobe}, top-{wl['k']}", "N": wl["N"], "nlist": wl["nlist"], "batch": wl["batch"], "nprobe": nprobe,
            "k": wl["k"], "parallelism": f"list-range shards x{n_gpus}" if n_gpus > 1 else "1 gpu",
            "l2": (f"index ({per_gpu_gb:.1f} GB of codes per GPU) is larger than L2; every step uses a different query batch" if per_gpu_gb > 0.2 else
                   f"index ({per_gpu_gb * 1000:.0f} MB of codes) fits L2: a latency case, not a bandwidth case")}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1412.0}, "fallback"


def csrc_sha():
    """Hash of the CUDA sources: ties an ncu-derived number under profiles/ to the tree it was measured on."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "densephrases_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            h.update(f.encode()); h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


class ClockSampler:
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.p = gpu, None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.gpu)],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self, t0=None, t1=None):
        """Summary over samples whose timestamp falls inside [t0, t1] (time.time() seconds) when given."""
        import datetime
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out = self.p.communicate(timeout=5)[0]
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if t0 is not None and not (t0 - 0.02 <= ts <= t1 + 0.02):
                    continue
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v == "Active":
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "samples": len(sm),
                "reasons": sorted(reasons)}


# ---- queries: identical in both arms ------------------------------------------------------------------------------------------
def make_query_plan(wl, nbatches):
    """SURVEY 8d 'near' queries: q = A^T (centroid + decode(code_j)) + N(0, 0.3^2) for random stored vectors j.  The random part
    (which vectors, which noise) comes from one seeded CPU generator; `finish_queries` turns it into vectors given the
    reconstructed rows, which each arm gets from its own index (bit-identical by tests/test_search_gpu.py)."""
    import torch
    g = torch.Generator().manual_seed(SEED_QUERY)
    total = nbatches * wl["batch"]
    ids = torch.randint(0, wl["N"], (total,), generator=g, dtype=torch.int64)
    noise = torch.randn((total, D), generator=g, dtype=torch.float32) * 0.3
    return ids, noise


def finish_queries(v, noise, A):
    """v [m,768] fp32 reconstructed rows (rotated space), A the OPQ matrix -> q = v A + noise, the product in fp64 on the host so
    that the GPU arm and the CPU arm get the same fp32 bits from the same rows."""
    import torch
    try:                                   # torchrun exports OMP_NUM_THREADS=1: give this one-off fp64 product a fair share of the host
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    torch.set_num_threads(max(1, cores // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1"))))))
    q = (v.double() @ torch.from_numpy(A).double()).float() + noise
    return q.contiguous()


def ref_index_for(wl, oracle):
    A = opq_matrix(SEED_INDEX)
    return oracle.RefIndex(A, oracle.gen_pq(SEED_INDEX), wl["lens"], centroids=oracle.gen_centroids(SEED_INDEX, 0, wl["nlist"]), seed=SEED_INDEX)


def oracle_threads(oracle):
    """All host cores, also under torchrun (which exports OMP_NUM_THREADS=1 to every rank)."""
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    oracle.lib().ref_set_num_threads.argtypes = [__import__("ctypes").c_int]
    oracle.lib().ref_set_num_threads(cores)
    return int(oracle.lib().ref_num_threads())


def cpu_search(ref, x, k, nprobe, resident_budget_gb=48.0, repeats=1):
    """The oracle (FAISS-equivalent CPU restatement, OpenMP over queries like faiss parallel_mode 0) on queries x.  The lists the
    sample probes are materialised in RAM first (faiss scans resident inverted lists; generated in parallel = parallel first
    touch), untimed.  -> (seconds per pass [repeats], D, I, note, probed GB)"""
    xr = ref.rotate(x)
    _, key = ref.coarse(xr, nprobe)
    lists = np.unique(key[key >= 0])
    need_gb = float(ref.list_len[lists].sum()) * 96 / 1e9
    rr, note = ref, f"lists regenerated on the fly ({need_gb:.1f} GB over the RAM budget)"
    if need_gb <= resident_budget_gb:
        rr, note = ref.with_resident_lists(lists), f"{need_gb:.1f} GB of probed lists resident in RAM"
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        xr = rr.rotate(x)
        _, key = rr.coarse(xr, nprobe)
        Dr, Ir = rr.search_preassigned(xr, key, k)
        times.append(time.perf_counter() - t0)
    return times, Dr, Ir, note, need_gb


def bits_equal(Da, Ia, Db, Ib):
    return bool(np.array_equal(np.asarray(Da).view(np.int32), np.asarray(Db).view(np.int32)) and np.array_equal(Ia, Ib))


# ---- reference arm ------------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch
    from oracle import ivfpq_ref as oracle
    oracle.build()
    cores = oracle_threads(oracle)
    torch.set_num_threads(max(1, min(cores, 32)))
    wl = workload_for(args.gpus, args.scale)
    W, K = args.warmup, args.steps
    ref = ref_index_for(wl, oracle)
    # bounded sample: the first nq queries of each batch the GPU arm times (whole batch at C2; `cores` queries of 1024 at C4)
    nq = min(wl["batch"], max(64, cores))
    ids, noise = make_query_plan(wl, W + K)
    sel = np.concatenate([np.arange(s * wl["batch"], s * wl["batch"] + nq) for s in range(W + K)])
    v, _ = ref.reconstruct(ids.numpy()[sel])
    X = finish_queries(torch.from_numpy(v), noise[sel], ref.A).numpy().reshape(W + K, nq, D)

    def probed(x):
        _, key = ref.coarse(ref.rotate(x), wl["nprobe"])
        lists = np.unique(key[key >= 0])
        return lists, float(ref.list_len[lists].sum()) * 96 / 1e9
    # faiss scans RAM-resident inverted lists: materialise what the sample probes (generated by all cores = parallel first touch).
    # If the lists of all W+K batches do not fit the budget, every step re-runs the sample of the LAST timed batch.
    budget = 64.0
    lists, need_gb = probed(X.reshape(-1, D))
    distinct = need_gb <= budget
    if not distinct:
        X = np.broadcast_to(X[W + K - 1], X.shape)
        lists, need_gb = probed(X[0])
    rr = ref.with_resident_lists(lists) if need_gb <= budget else ref
    times = []
    for s in range(W + K):
        t0 = time.perf_counter()
        xr = rr.rotate(X[s])
        _, key = rr.coarse(xr, wl["nprobe"])
        rr.search_preassigned(xr, key, wl["k"])
        times.append(time.perf_counter() - t0)
    t = sum(times[W:])
    qps = nq * K / t
    sample = (f"{nq} of the {wl['batch']} queries of " + ("each timed batch" if distinct else "the last timed batch, repeated every step") +
              f" (the GPU arm's own query vectors), full nprobe={wl['nprobe']} scan over " +
              (f"RAM-resident inverted lists ({need_gb:.1f} GB probed)" if rr is not ref else "lists regenerated on the fly") +
              f", OpenMP over queries on {cores} threads")
    # C1 (BASELINE.json configs[0]): the reference's own CPU-runnable case
    c1 = c1_cpu(oracle, cores)
    # C3 (configs[2]) on the host, N = 1 only (the GPU arm reports it in `encoder.c3`)
    c3 = c3_cpu(oracle, cores, wl, ref) if args.gpus == 1 else None
    line = {"impl": "reference", "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": args.gpus,
            "steps": K, "warmup": W, "ms_per_step": 1000.0 * t / K, "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(wl, args.gpus), "where": "host cpu",
            "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "step_ms_min_max": [1000.0 * min(times[W:]), 1000.0 * max(times[W:])], "c1": c1}
    if c3 is not None:
        line["c3"] = c3
    emit(line)
    return 0


def c3_cpu(oracle, cores, wl, ref):
    """C3 on the host: 64 questions (the GPU arm's token ids and weights: same seeds) -> both towers under torch on the CPU cores
    (oracle/encoder_ref.py, the restatement pinned to the reference Encoder: the reference's own path is torch eager fp32,
    single_utils.py:116) -> ONE stacked 128-vector search of the C2 index by the FAISS-equivalent restatement."""
    import torch
    from densephrases_b200.encoder import BertGeometry, random_state_dict, synthetic_query_batch      # seeded data generators only
    from oracle import encoder_ref
    geo = BertGeometry()
    sd = random_state_dict(geo, 1)
    ids, mask, tt = synthetic_query_batch(64, 64, geo.vocab_size, 2)
    best = None
    for threads in sorted({max(1, min(cores, 32)), max(1, cores)}):       # MKL does not always scale to every core: keep the better setting
        torch.set_num_threads(threads)
        encoder_ref.embed_query(sd, ids[:4], mask[:4], tt[:4])
        t0 = time.perf_counter()
        s, e = encoder_ref.embed_query(sd, ids, mask, tt)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, threads)
    t_enc, enc_threads = best
    x = torch.cat([s[:, 0], e[:, 0]], 0).numpy()
    xr = ref.rotate(x)
    _, key = ref.coarse(xr, wl["nprobe"])
    lists = np.unique(key[key >= 0])
    need_gb = float(ref.list_len[lists].sum()) * 96 / 1e9
    rr = ref.with_resident_lists(lists) if need_gb <= 64.0 else ref
    t0 = time.perf_counter()
    xr = rr.rotate(x)
    _, key = rr.coarse(xr, wl["nprobe"])
    rr.search_preassigned(xr, key, wl["k"])
    t_search = time.perf_counter() - t0
    return {"questions_per_s": 64.0 / (t_enc + t_search), "ms_per_64_questions": 1000.0 * (t_enc + t_search),
            "encoder_ms": 1000.0 * t_enc, "encoder_threads": enc_threads, "search_ms": 1000.0 * t_search, "search_threads": cores, "kind": "port",
            "what": "64 questions: both towers under torch fp32 on the host cores + one stacked 128-vector search on the C2 index "
                    f"({need_gb:.1f} GB of probed lists resident in RAM)"}


def c1_cpu(oracle, cores, x=None):
    """C1: FAISS-CPU IVF1,PQ96 flat index, 1M phrases, 100 queries (nprobe_eff = 1): the CPU restatement on all cores."""
    import torch
    wl = workload("C1")
    ref = ref_index_for(wl, oracle)
    if x is None:
        ids, noise = make_query_plan(wl, 1)
        v, _ = ref.reconstruct(ids.numpy())
        x = finish_queries(torch.from_numpy(v), noise, ref.A).numpy()
    times, Dr, Ir, note, _ = cpu_search(ref, x, wl["k"], wl["nprobe"], repeats=4)
    t = min(times[1:])
    return {"workload": config_dict(wl, 1)["workload"], "value": wl["batch"] / t, "unit": "queries/s", "cores": cores, "kind": "port",
            "ms_per_batch": 1000.0 * t, "note": note, "_D": Dr, "_I": Ir}


# ---- our arm ------------------------------------------------------------------------------------------------------------------
class Ctx:
    pass


def timed_loop(cx, fn, steps):
    """W untimed + exactly K timed calls of fn(s), barrier + synchronize on both sides, CUDA events, max over ranks."""
    import torch
    W, K = cx.W, cx.K
    for s in range(W):
        fn(s)
    cx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cx.barrier()
    t0 = time.time()
    e0.record()
    out = None
    for s in range(W, W + K):
        out = fn(s)
    e1.record()
    cx.barrier()
    t1 = time.time()
    return cx.max_over_ranks(e0.elapsed_time(e1)), out, (t0, t1)


def measure_search(cx, ix, wl, Q, Qh, nprobe, sample_clocks=False):
    """One full measurement of the sharded/unsharded search at `nprobe`: device-resident value, end-to-end through the host API,
    roofline of the scan kernel, algorithmic bytes.  Returns a dict (rank 0 uses it)."""
    import torch
    W, K, k = cx.W, cx.K, wl["k"]
    ix.nprobe = nprobe
    B = wl["batch"]
    sampler = cx.sampler if (sample_clocks and cx.rank == 0) else None      # started at process start: nvidia-smi needs time to warm up
    ms_dev, last, (tw0, tw1) = timed_loop(cx, lambda s: ix.search_device(Q[s], k), K)
    clocks = sampler.stop(tw0, tw1) if sampler else None
    last_dev = (last[0].cpu().numpy(), last[1].cpu().numpy())
    cx.stage(f"{wl['name']} nprobe {nprobe}: device pass {ms_dev / K:.3f} ms/step")
    ms_e2e, last_h, _ = timed_loop(cx, lambda s: ix.search(Qh[s] if cx.world > 1 else Qh[s].numpy(), k), K)
    assert bits_equal(last_h[0], last_h[1], last_dev[0], last_dev[1]), "host-API results differ from the device-resident results"
    cx.stage(f"{wl['name']} nprobe {nprobe}: e2e pass {ms_e2e / K:.3f} ms/step")

    # roofline of the dominant kernel (PQ scan): (a) algorithmic bytes of each timed batch on this rank (untimed pass),
    # (b) the same K steps back to back with CUDA events around the scan kernel on the launching stream
    lens = wl["lens"]
    lo, hi = ix.range
    local = ix.local
    nsteps = min(K, 60)
    alg_bytes = []

    def one(s):
        if cx.world > 1:
            ix.search_device(Q[s], k)
        else:
            local.search(Q[s], k)
    for s in range(W + K - nsteps, W + K):
        one(s)
        pr = local.last_probes(B).astype(np.int64)
        m = (pr >= lo) & (pr < hi)
        alg_bytes.append(float(lens[pr[m]].sum()) * 96.0)
    local.set_profile(True)
    cx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(W + K - nsteps, W + K):
        one(s)
    e1.record()
    torch.cuda.synchronize()
    ms_prof_pass = e0.elapsed_time(e1)
    scan_ms = [float(v) for v in local.profile_scan_ms()][-nsteps:]
    local.set_profile(False)
    flags = int(local.last_flags(B).sum())
    group = local.last_group_size()
    pair_mode = group > 1
    pk, pk_kind = peaks()
    t_scan = sum(scan_ms) / len(scan_ms) / 1000.0
    mean_bytes = sum(alg_bytes) / len(alg_bytes)
    achieved = mean_bytes / t_scan / 1e9 if t_scan > 0 else 0.0
    kernel = {1: "scan_kernel<FAST>", 2: "scan_pair_kernel", 4: "scan_quad_kernel"}[group]
    traffic, tsrc = lookup_traffic(kernel, wl["name"], nprobe, cx.world)
    roofline = {"kernel": kernel, "gathers": {1: "one query per gather (fp32 LUT)", 2: "two queries per gather (pair-packed u16 LUTs)", 4: "four queries per gather (quad-packed u8 LUTs)"}[group],
                "bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"], "peak_kind": pk_kind,
                "traffic": traffic, "traffic_source": tsrc, "kernel_ms": 1000.0 * t_scan, "algorithmic_bytes_per_launch": mean_bytes,
                "share_of_step": 1000.0 * t_scan / (ms_prof_pass / nsteps), "step_ms_same_pass": ms_prof_pass / nsteps,
                "how": f"CUDA events around the kernel inside a back-to-back {nsteps}-step loop on the launching stream (rank 0's shard)"}
    if pair_mode:
        roofline["note"] = ("algorithmic bytes count every (query, probed vector) pair; the kernel serves the 2 / 4 queries of a group from one code read and "
                            "later readers of a list from L2, so achieved > DRAM traffic and frac may exceed 1; the kernel's own limiters are the LSU "
                            "data pipe (shared-memory gathers) and the issue slots, see profiles/ and DESIGN.md 4.1")
    # step-level fraction of the HBM roofline: all ranks' algorithmic bytes / (step time x N x peak)
    tot_bytes = cx.sum_over_ranks(mean_bytes)
    step_frac = tot_bytes / (ms_dev / K / 1000.0) / 1e9 / (cx.world * pk["hbm_gbs"])
    # kernels of this repo launched per search step (counted from the per-launch lists in profiles/: r2q_launches_c2.csv,
    # r2q_launches_shard_c4_np*.csv): one GPU: rotation, coarse quantizer, tables, plan, scan, merge, 4 early-exit fallback launches;
    # sharded: + record pack / unpack (query-split) or coarse merge (list-split), + top-k pack and merge
    from densephrases_b200.sharded import use_query_split
    if cx.world == 1:
        launches = 18 if pair_mode else 12
    elif use_query_split(B, cx.world, wl["nlist"]):
        launches = 26 if pair_mode else 21
    else:
        launches = 21 if pair_mode else 15
    return {"nprobe": nprobe, "value": B * K / (ms_dev / 1000.0), "ms_per_step": ms_dev / K,
            "e2e": {"value": B * K / (ms_e2e / 1000.0), "unit": "queries/s", "h2d_bytes_per_step": B * D * 4, "d2h_bytes_per_step": B * k * 12,
                    "ms_per_step": ms_e2e / K},
            "roofline": roofline, "step_frac_of_hbm_roofline": step_frac, "hbm_roofline_qps": B / (tot_bytes / (cx.world * pk["hbm_gbs"] * 1e9)),
            "gpu_launches_per_step": launches, "exact_fallback_queries_last_batch": flags, "clocks": clocks,
            "_last": last_dev}


def lookup_traffic(kernel, wl_name, nprobe, world):
    """dram bytes per launch of `kernel` from the ncu pass tools/profile.sh made on THIS tree (profiles/traffic.json, keyed by the
    hash of csrc/); null when the sources changed since."""
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(tp):
        return None, "no profiles/traffic.json"
    tj = json.load(open(tp))
    if tj.get("csrc_sha") != csrc_sha():
        return None, f"profiles/traffic.json was measured on csrc {tj.get('csrc_sha')}, this tree is {csrc_sha()}"
    key = f"{kernel}|{wl_name}|nprobe{nprobe}|n{world}"
    ent = tj.get("entries", {}).get(key)
    if not ent:
        return None, f"no ncu capture for {key}"
    return ent.get("dram_bytes_per_launch"), {"file": "profiles/traffic.json", "csrc_sha": tj["csrc_sha"], "ncu_report": ent.get("report"),
                                              "limiter": ent.get("limiter")}


OC_KEYS = ("queries", "identical_ids_and_fp32_scores", "max_abs_score_minus_fp64_decoded_dot", "all_labels_found", "cpu_seconds", "cores", "note")


def oracle_check(cx, wl, nprobe, Qh_last, last_dev, nq):
    """Rank 0: `nq` sampled queries of the last timed batch through the CPU oracle (probed lists regenerated from the seed),
    compared bit for bit with what the GPUs returned.  Also the timed cpu_baseline at N=1."""
    from oracle import ivfpq_ref as oracle
    oracle.build()
    cores = oracle_threads(oracle)
    ref = ref_index_for(wl, oracle)
    step = max(1, wl["batch"] // nq)
    pick = np.arange(0, wl["batch"], step)[:nq]
    x = Qh_last[pick].numpy()
    times, Dr, Ir, note, gb = cpu_search(ref, x, wl["k"], nprobe)
    same = bits_equal(Dr, Ir, last_dev[0][pick], last_dev[1][pick])
    # decoded-vector check (SURVEY 8c identity): every returned score equals <A x, centroid + decode(code)> in fp64 up to fp32 rounding
    Dg, Ig = last_dev[0][pick], last_dev[1][pick]
    ok = Ig >= 0
    v, found = ref.reconstruct(Ig[ok])
    xr64 = (ref.A.astype(np.float64) @ x.astype(np.float64).T).T                      # [nq, 768]
    rows = np.nonzero(ok)[0]
    dots = np.einsum("ij,ij->i", v.astype(np.float64), xr64[rows])
    dec_err = float(np.abs(dots - Dg[ok].astype(np.float64)).max()) if len(dots) else 0.0
    return {"queries": int(len(pick)), "identical_ids_and_fp32_scores": same, "cpu_seconds": times[0], "cores": cores, "note": note,
            "qps": len(pick) / times[0], "max_abs_score_minus_fp64_decoded_dot": dec_err, "all_labels_found": bool(found.all())}


def run_ours(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from densephrases_b200.sharded import ShardedIvfPq

    T0 = time.time()
    cx = Ctx()
    cx.rank, cx.world, cx.local_rank, cx.dev, cx.W, cx.K = rank, world, local_rank, dev, args.warmup, args.steps

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        import torch.distributed as dist
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v):
        if world == 1:
            return v
        import torch.distributed as dist
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def stage(msg):
        if rank == 0 and args.verbose:
            print(f"[bench +{time.time() - T0:.1f}s] {msg}", file=sys.stderr, flush=True)
    cx.barrier, cx.max_over_ranks, cx.sum_over_ranks, cx.stage = barrier, max_over_ranks, sum_over_ranks, stage

    def build(wl):
        ix = ShardedIvfPq(wl["nlist"], rank=rank, world=world, device=local_rank)
        ix.build_synthetic(opq_matrix(SEED_INDEX), wl["lens"], SEED_INDEX)
        torch.cuda.synchronize()
        return ix

    def queries(ix, wl, nb):
        ids, noise = make_query_plan(wl, nb)
        v, _ = ix.local.reconstruct_batch(ids.to(dev))
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(v)               # every label lives on exactly one shard, the others contribute zero rows
        Qh = finish_queries(v.cpu(), noise, ix.local.opq_matrix()).reshape(nb, wl["batch"], D).pin_memory()
        return Qh.to(dev), Qh

    wl = workload_for(world, args.scale)
    W, K = cx.W, cx.K
    cx.sampler = None
    if rank == 0:
        cx.sampler = ClockSampler(local_rank)
        cx.sampler.start()
    ix = build(wl)
    Q, Qh = queries(ix, wl, W + K)
    stage(f"{wl['name']} index built ({ix.local.device_bytes / 1e9:.1f} GB on this rank), queries made")
    main = measure_search(cx, ix, wl, Q, Qh, wl["nprobe"], sample_clocks=True)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, *main["_last"])
    second = None
    if wl["name"] == "C4":
        second = measure_search(cx, ix, wl, Q, Qh, 32)
    line = None
    if rank == 0:
        line = {"metric": METRIC, "value": main["value"], "unit": "queries/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config_dict(wl, world), "where": "hbm", "e2e": main["e2e"],
                "gpu_launches": K * main["gpu_launches_per_step"], "roofline": main["roofline"],
                "step_frac_of_hbm_roofline": main["step_frac_of_hbm_roofline"], "hbm_roofline_qps": main["hbm_roofline_qps"], "clocks": main["clocks"],
                "exact_fallback_queries_last_batch": main["exact_fallback_queries_last_batch"], "csrc_sha": csrc_sha()}
        if world > 1:
            line["scaling_note"] = ("strong scaling: C4's 1B-phrase index and batch 1024 are fixed for every N >= 2; the N = 1 line is C2 and carries "
                                    "C4 on one GPU in its `c4_1gpu` object")
        if not args.no_cpu:
            # N = 1: the timed cpu_baseline (64 queries = the whole last batch); N > 1: 16 sampled queries checked against the oracle
            nq = min(wl["batch"], 64) if world == 1 else 16
            oc = oracle_check(cx, wl, wl["nprobe"], Qh[W + K - 1], main["_last"], nq)
            if world == 1:
                line["cpu_baseline"] = {"value": oc["qps"], "unit": "queries/s", "cores": oc["cores"], "kind": "port",
                                        "sample": f"{oc['queries']} queries of the last timed batch, full nprobe={wl['nprobe']} scan, {oc['note']}; "
                                                  f"GPU results bit-identical: {oc['identical_ids_and_fp32_scores']}"}
            else:
                line["cpu_baseline"] = None
            line["oracle_check"] = {k_: oc[k_] for k_ in OC_KEYS}
        if second is not None:
            s2 = {k_: v for k_, v in second.items() if not k_.startswith("_") and k_ != "clocks"}
            s2["config"] = config_dict(wl, world, 32)
            if not args.no_cpu:
                oc2 = oracle_check(cx, wl, 32, Qh[W + K - 1], second["_last"], 16)
                s2["oracle_check"] = {k_: oc2[k_] for k_ in OC_KEYS}
            line["nprobe32"] = s2
    if world > 1:
        barrier()

    # ---- N = 1 only: the other configs of BASELINE.json in the same line ----
    if world == 1:
        if not args.no_encoder:
            line["encoder"] = encoder_leg(cx, ix, wl)
            stage("encoder leg done")
        del ix, Q
        torch.cuda.empty_cache()
        if not args.no_c1:
            line["c1"] = c1_leg(cx, build, queries, args)
            stage("C1 leg done")
        if not args.no_c4:
            line["c4_1gpu"] = c4_single_gpu_leg(cx, build, queries, args)
            stage("C4 on one GPU done")
    else:
        del ix
    if rank == 0:
        emit(line)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


def dump_outputs(out_dir, D, I):
    """What the last timed step of the headline search returned to its caller: top-k scores (fp32) and labels (int64, stored as
    float64, exact below 2^53), each [batch, k].  The queries are seeded, so two builds run with the same arguments can be compared."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "scores.npy"), np.asarray(D, dtype=np.float32))
    np.save(os.path.join(out_dir, "labels.npy"), np.asarray(I).astype(np.float64))


def c1_leg(cx, build, queries, args):
    """C1 (BASELINE.json configs[0]): IVF1,PQ96, 1M phrases, 100 queries -- the reference's own CPU-runnable case, on the GPU and
    through the CPU oracle on the same 100 queries."""
    import torch
    wl = workload("C1")
    ix = build(wl)
    Q, Qh = queries(ix, wl, 1)           # the same 100 queries as the reference arm's C1 leg
    ix.nprobe = wl["nprobe"]
    k = wl["k"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        Dd, Id = ix.search_device(Q[0], k)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(20):
        Dd, Id = ix.search_device(Q[0], k)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 20
    t0 = time.perf_counter()
    for _ in range(10):
        Dh, Ih = ix.search(Qh[0].numpy(), k)
    ms_e2e = (time.perf_counter() - t0) * 100.0
    out = {"workload": config_dict(wl, 1)["workload"], "gpu": {"value": wl["batch"] / ms * 1000.0, "unit": "queries/s", "ms_per_batch": ms,
                                                              "e2e_value": wl["batch"] / ms_e2e * 1000.0, "queries_per_gather": ix.local.last_group_size()}}
    if not args.no_cpu:
        from oracle import ivfpq_ref as oracle
        oracle.build()
        cores = oracle_threads(oracle)
        c = c1_cpu(oracle, cores, Qh[0].numpy())
        same = bits_equal(c.pop("_D"), c.pop("_I"), Dh, Ih)
        c.pop("workload")
        out["cpu"] = c
        out["gpu_results_bit_identical_to_cpu"] = same
    return out


def c4_single_gpu_leg(cx, build, queries, args):
    """C4's index (1B phrases, IVF65536, 96 GB of codes) held by ONE B200, batch 1024: the N = 1 point of the metric's 1/2/4/8 series."""
    import torch
    wl = workload("C4", args.scale)
    ix = build(wl)
    Q, Qh = queries(ix, wl, cx.W + cx.K)
    out = {"steps": cx.K, "warmup": cx.W}
    for nprobe in (wl["nprobe"], 32):
        m = measure_search(cx, ix, wl, Q, Qh, nprobe)
        r = {k_: v for k_, v in m.items() if not k_.startswith("_") and k_ != "clocks"}
        r["config"] = config_dict(wl, 1, nprobe)
        if not args.no_cpu:
            oc = oracle_check(cx, wl, nprobe, Qh[cx.W + cx.K - 1], m["_last"], 16)
            r["oracle_check"] = {k_: oc[k_] for k_ in OC_KEYS}
        out[f"nprobe{nprobe}"] = r
    del ix
    torch.cuda.empty_cache()
    return out


def encoder_leg(cx, ix, wl):
    """C3: query encoder (2 x SpanBERT-base towers, random-init weights, synthetic tokens) alone in each precision mode, the
    reference's own torch path (oracle/encoder_ref.py = HF-BERT restatement pinned to the unmodified reference Encoder) on the
    same GPU as the baseline, and encoder -> search end to end from host token ids to host results."""
    import torch
    from densephrases_b200.encoder import BertGeometry, Encoder, random_state_dict, synthetic_query_batch
    dev, k = cx.dev, wl["k"]
    pk, _ = peaks()
    geo = BertGeometry()
    sd = random_state_dict(geo, 1)
    enc = Encoder(geo, state_dict=sd, device=cx.local_rank)
    ids_h, mask_h, tt_h = (t.pin_memory() for t in synthetic_query_batch(64, 64, geo.vocab_size, 2))
    ids, mask, tt = (t.to(dev) for t in (ids_h, mask_h, tt_h))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    flops = 64 * 22.05e9
    tf32_peak = pk["bf16_tflops"] / 2.0
    tf32_sustained = pk.get("bf16_tflops_sustained", pk["bf16_tflops"]) / 2.0
    info = {"note": "B=64,S=64; 22.05 GFLOP/question over both towers (SURVEY 8a a6); TF32 peak taken as half the measured bf16 peak"}

    def time_fn(fn, reps=20, warm=5):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps, out

    outs = {}
    for mode in enc.precision_modes():
        enc.set_precision(mode)
        ms, o = time_fn(lambda: enc.embed_query(ids, mask, tt))
        outs[mode] = torch.cat([o[0][:, 0], o[1][:, 0]], 0).clone()
        mult = enc.mma_multiplier(mode)
        info[mode] = {"ms_per_64_questions": ms, "questions_per_s": 64000.0 / ms, "algorithmic_tflops": flops / ms / 1e9,
                      "mma_tflops_issued_tf32_equivalent": flops * mult / ms / 1e9,
                      "tensor_pipe_frac_of_tf32_peak_burst": flops * mult / ms / 1e9 / tf32_peak,
                      "tensor_pipe_frac_of_tf32_peak_sustained": flops * mult / ms / 1e9 / tf32_sustained}
    # the reference's own path under torch on this GPU (fp32 eager; TF32 matmuls off and on), same weights, same tokens
    try:
        from oracle import encoder_ref
        sd_gpu = {k_: v_.to(dev) for k_, v_ in sd.items()}
        for name, allow in (("torch_fp32", False), ("torch_tf32", True)):
            torch.backends.cuda.matmul.allow_tf32 = allow
            torch.backends.cudnn.allow_tf32 = allow
            ms, o = time_fn(lambda: encoder_ref.embed_query(sd_gpu, ids, mask, tt), reps=5, warm=2)
            r = torch.cat([o[0][:, 0], o[1][:, 0]], 0)
            info[name] = {"ms_per_64_questions": ms, "questions_per_s": 64000.0 / ms, "algorithmic_tflops": flops / ms / 1e9}
            if name == "torch_fp32":
                ref_out = r.clone()
        torch.backends.cuda.matmul.allow_tf32 = False
        for mode, o in outs.items():
            info[mode]["max_abs_diff_vs_torch_fp32"] = float((o - ref_out).abs().max())
        info["torch_tf32"]["max_abs_diff_vs_torch_fp32"] = float((r - ref_out).abs().max())
        del sd_gpu
    except Exception as ex:      # the torch arm is a baseline, never a dependency of the product path
        info["torch_baseline_error"] = repr(ex)
    # C3 end to end in the mode that meets the 1e-3 tolerance: 64 questions (host token ids) -> encoder -> ONE stacked [128,768]
    # search (start rows then end rows, index.py:195-202) -> host (D, I)
    mode = enc.default_mode()
    enc.set_precision(mode)
    ix.nprobe = wl["nprobe"]
    Dh = torch.empty((128, k), dtype=torch.float32).pin_memory()
    Ih = torch.empty((128, k), dtype=torch.int64).pin_memory()

    def c3():
        a, b, c = ids_h.to(dev, non_blocking=True), mask_h.to(dev, non_blocking=True), tt_h.to(dev, non_blocking=True)
        qs, qe = enc.embed_query(a, b, c)
        Dd, Id = ix.search_device(torch.cat([qs[:, 0], qe[:, 0]], 0).contiguous(), k)
        Dh.copy_(Dd, non_blocking=True); Ih.copy_(Id, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    ms, _ = time_fn(c3, reps=10, warm=3)
    info["c3"] = {"mode": mode, "questions_per_s": 64000.0 / ms, "ms_per_64_questions": ms, "h2d_bytes_per_step": 3 * 64 * 64 * 8,
                  "d2h_bytes_per_step": 128 * k * 12, "what": "host token ids -> 2 towers -> stacked 128-vector search on the C2 index -> host top-10"}
    del enc
    return info


_REAL_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout; NCCL prints a version banner there (seen on the GPU box).  Route fd 1 to stderr for
    the whole run and keep the real stdout for the final line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _clean(o):
    if isinstance(o, dict):
        return {k: _clean(v) for k, v in o.items() if not str(k).startswith("_")}
    if isinstance(o, (list, tuple)):
        return [_clean(v) for v in o]
    if isinstance(o, (np.floating, np.integer)):
        return o.item()
    if isinstance(o, np.bool_):
        return bool(o)
    return o


def emit(line):
    data = (json.dumps(_clean(line)) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="default: 100 (ours), 10 (--impl reference: each step is seconds of all-core CPU work)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="debug only: shrink the number of phrases (the headline run uses 1.0)")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / oracle-check legs")
    ap.add_argument("--no-encoder", action="store_true", help="skip the C3 encoder leg")
    ap.add_argument("--no-c1", action="store_true", help="skip the C1 leg")
    ap.add_argument("--no-c4", action="store_true", help="N=1: skip the C4-on-one-GPU leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the top-k scores and labels of the last timed step of the headline search to DIR/{scores,labels}.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.steps is None:
        args.steps = 10 if args.impl == "reference" else 100
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records this repo's CUDA path (--impl ours)")
    quiet_stdout()
    return run_reference(args) if args.impl == "reference" else run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
