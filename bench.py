#!/usr/bin/env python
"""bench.py -- queries/sec of SearchArray's scoring hot path on B200 (see BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # the CPU reference arm
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR   # + the last timed step's top-k as .npy

Workload (config.workload): BASELINE.json configs[1] -- 10M-doc synthetic MSMARCO-shaped corpus
(searcharray_b200/synth.py, seeded, generated as postings), single-term BM25.  One "step" = one
pass over a batch of `--queries` (1,024) DISTINCT stratified single-term queries: every query
produces the dense float32[N] BM25 score vector in HBM and its exact top-k.  For N > 1 the 10M docs
are sharded by contiguous doc-id range (strong scaling), one process per GPU, one ncclAllGather of
the per-shard top-k per batch.

  value : device-resident throughput -- query descriptors already in HBM, CUDA events on the
          library's stream around exactly K x sa_batch_execute (kernels + all-gather), max over ranks.
  e2e   : the same batch through the public C-ABI call with HOST buffers per step
          (sa_score_batch_topk: H2D of the query descriptors, kernels, D2H of the top-k).
  e2e_dense : the literal `.score()` drop-in (sa_score_term), D2H of the dense float32[N] per query.
  roofline  : term_tile_kernel, algorithmic bytes 8*W + 4*df + 4*N per query (SURVEY 8d) over the
          kernel's CUDA-event time, against MEASURED_PEAKS.json's hbm_gbs; per-df-bucket fractions.
  cpu_baseline : the reference's own `SearchArray.score` (oracle/_ref, `kind: "reference"`; the
          oracle port when that build is absent) on the host cores, bounded sample, NO top-k
          (the reference's stock call returns the dense vector; a top-k variant is reported apart).
  verify : GPU top-k (docs AND score bits) of a sample of the step's queries against the CPU oracle.
Extra blocks: `phrase` (configs[2]; rare-term and hard strata, B_phrase roofline), `phrase.slop2`
(configs[3]), `bigram` (BASELINE.md's common x mid case), `edismax` (configs[4] shape).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K1, B = 1.2, 0.75


def log(*a):
    if int(os.environ.get("RANK", "0")) == 0:
        print("[bench]", *a, file=sys.stderr, flush=True)


def dbg(*a):
    """progress marks of EVERY rank (SA_BENCH_DEBUG=1): where a multi-rank run is, should it ever stall"""
    if os.environ.get("SA_BENCH_DEBUG"):
        print(f"[bench r{os.environ.get('RANK', '0')} +{time.time() % 1000:.1f}s]", *a, file=sys.stderr, flush=True)


# --------------------------------------------------------------------------- corpus
def build_corpus(n_docs, rank, world, field="body"):
    from searcharray_b200 import synth
    spec = synth.SynthSpec(n_docs, field=field)
    t0 = time.time()
    host, lo, hi = synth.generate_shard(spec, rank, world)
    avgdl = synth.global_avg_doc_length(spec)       # float32 of the exact global mean, same on every rank
    log(f"rank {rank}: {field} docs [{lo},{hi}) {host.words.nbytes / 1e6:.0f} MB of postings, "
        f"{host.n_terms} terms, in {time.time() - t0:.1f}s, avgdl={avgdl}")
    return spec, host, lo, hi, avgdl


def make_queries(spec, n_queries):
    from searcharray_b200 import synth
    names = synth.stratified_term_queries(spec, n_queries)
    return names, np.asarray([spec.term_index[n] for n in names], dtype=np.uint32)


def idf_of(n_docs, df):
    from searcharray_b200.similarity import compute_idf
    return np.asarray([compute_idf(n_docs, np.asarray([d])) for d in df], dtype=np.float32)


def phrase_idf(n_docs, df, term_ids):
    d = df[np.asarray(term_ids)].astype(np.float64)
    return np.float32(np.sum(np.log(1 + (n_docs - d + 0.5) / (d + 0.5))))


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "25"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def count_since(self, t_from):
        return sum(1 for t, _ in self.lines if t >= t_from)

    def stop(self, t_from=0.0, t_to=None):
        """Summary of the samples taken in [t_from, t_to] (the timed regions)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, ln in self.lines:
            if t < t_from or (t_to is not None and t > t_to):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------- CPU reference arm
class CpuArm:
    """The reference's CPU path for this workload: its own SearchArray.score (oracle/_ref, built from
    /root/reference by oracle/build_ref.py) over the injected synthetic index; the oracle port
    (oracle/search.py, the same algorithm restated in C + numpy) when that build is absent."""

    def __init__(self, spec, host, avgdl, n_docs):
        from oracle import ref_runner
        self.spec, self.host = spec, host
        self.names = [t[0] for t in spec.terms]
        if ref_runner.available() and not os.environ.get("SA_BENCH_FORCE_PORT"):
            self.kind = "reference"
            self.arr = ref_runner.reference_array(host, avg_doc_length=avgdl, corpus_size=n_docs, names=self.names)
            self.sim = ref_runner.bm25(K1, B)
        else:
            from oracle import search as osearch
            self.kind = "port"
            self.idx = osearch.OracleIndex({t: host.term_words(t) for t in range(host.n_terms)}, host.doc_lens,
                                           avg_doc_length=avgdl, corpus_size=n_docs, cache=True)

    def score_term(self, term_id):
        """SearchArray.score(term) (reference postings.py:652-680): the dense float32[N] vector."""
        if self.kind == "reference":
            return self.arr.score(self.names[int(term_id)], similarity=self.sim)
        return self.idx.score(int(term_id), k1=K1, b=B)

    def score_phrase(self, term_ids, slop=0):
        if self.kind == "reference":
            return self.arr.score([self.names[int(t)] for t in term_ids], similarity=self.sim, slop=slop)
        return self.idx.score([int(t) for t in term_ids], k1=K1, b=B, slop=slop)

    def warm(self, term_ids, threads=1):
        """tf / df caches of these terms, like SearchArray.index(autowarm=True) -> posns.warm()
        (reference middle_out.py:337-342) does at index time."""
        def one(t):
            if self.kind == "reference":
                self.arr.docfreq(self.names[int(t)])
                self.arr.posns.termfreqs(int(t))
            else:
                self.idx.docfreq(int(t))
                self.idx.termfreqs(int(t))
        uniq = [int(t) for t in np.unique(term_ids)]
        if threads > 1:
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(threads) as ex:
                list(ex.map(one, uniq))
        else:
            for t in uniq:
                one(t)

    def clear_cache(self):
        if self.kind == "reference":
            self.arr.posns.clear_cache()
        else:
            self.idx._df_cache.clear()
            self.idx._tf_cache.clear()


def run_cpu_sample(fn, items, threads):
    from concurrent.futures import ThreadPoolExecutor
    t0 = time.perf_counter()
    if threads == 1:
        for t in items:
            fn(t)
    else:
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(fn, items))
    return time.perf_counter() - t0


def best_thread_count(fn, term_ids, cores):
    """The reference's Cython loops release the GIL, so `.score` runs from a thread pool
    (test_msmarco.py:483-507); every call allocates a dense float32[N], so wide pools contend on
    the allocator / page faults.  Probe a few widths and keep the fastest: the baseline is the best
    the host can do with the stock call."""
    best, best_qps = 1, 0.0
    for th in sorted({1, 4, 8, 16, 32, 64, cores}):
        if th > cores:
            continue
        probe = term_ids[:min(len(term_ids), max(32, 2 * th))]
        dt = run_cpu_sample(fn, probe, th)
        qps = len(probe) / dt
        log(f"cpu probe: {th} threads -> {qps:.1f} qps")
        if qps > best_qps:
            best, best_qps = th, qps
    return best, best_qps


def cpu_topk(scores, k):
    """A sane top-k over the reference's dense vector (score desc, doc asc; score > 0)."""
    nz = np.flatnonzero(scores > 0)
    if len(nz) > k:
        part = np.argpartition(scores[nz], -k)[-k:]
        thr = scores[nz][part].min()
        nz = nz[scores[nz] >= thr]                      # keep ties so the doc-asc rule is exact
    order = np.lexsort((nz, -scores[nz].astype(np.float64)))[:k]
    return nz[order].astype(np.uint32), scores[nz[order]]


def cold_cpu_qps(arm, term_ids, n=6):
    """SURVEY 8d: the reference's COLD path (`posns.clear_cache()` before each query, as
    test_msmarco.py:362-379 does): tf by popcount and df by unique on every call.  One thread."""
    sample = [int(t) for t in term_ids[:n]]
    t0 = time.perf_counter()
    for t in sample:
        arm.clear_cache()
        arm.score_term(t)
    dt = time.perf_counter() - t0
    return {"value": len(sample) / dt, "unit": "queries/s", "cores": 1,
            "sample": f"{len(sample)} queries, tf/df caches cleared before each"}


def bench_reference(args, rank, world):
    if rank != 0:
        return                                  # rank 0 alone runs the CPU arm
    spec, host, lo, hi, avgdl = build_corpus(args.docs, 0, 1)
    names, term_ids = make_queries(spec, args.queries)
    cores = os.cpu_count() or 1
    arm = CpuArm(spec, host, avgdl, args.docs)
    t0 = time.time()
    arm.warm(term_ids, threads=min(cores, 32))
    log(f"reference arm ({arm.kind}): warmed tf/df caches of {len(np.unique(term_ids))} terms in {time.time() - t0:.1f}s")
    threads, probe_qps = best_thread_count(arm.score_term, term_ids, cores)
    # bounded sample: the whole --steps/--warmup run has to end within a few minutes
    budget_s = args.ref_budget
    per_step = int(probe_qps * budget_s / max(1, args.steps + args.warmup))
    q_step = len(term_ids) if per_step >= len(term_ids) else max(64, per_step // 64 * 64)
    sample = term_ids[:min(len(term_ids), q_step)]
    for _ in range(args.warmup):
        run_cpu_sample(arm.score_term, sample, threads)
    t = 0.0
    for _ in range(args.steps):
        t += run_cpu_sample(arm.score_term, sample, threads)
    qps = args.steps * len(sample) / t
    one_thread = len(sample[:32]) / run_cpu_sample(arm.score_term, sample[:32], 1)
    tk = sample[:24]
    topk_qps = len(tk) / run_cpu_sample(lambda q: cpu_topk(arm.score_term(q), args.k), tk, min(threads, 8))
    cold = cold_cpu_qps(arm, sample)
    line = {
        "impl": "reference", "metric": "queries/sec (single-term BM25 .score()) on 10M-doc synthetic MSMARCO",
        "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, len(sample)),
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "host_cores": cores, "kind": arm.kind,
                         "sample": f"{len(sample)} of the {args.queries} stratified term queries per step, stock "
                                   f"SearchArray.score (dense float32[N], no top-k), ThreadPool({threads}) = fastest "
                                   f"of the probed pool widths, warm tf/df caches",
                         "one_thread": {"value": one_thread, "unit": "queries/s"},
                         "score_plus_topk": {"value": topk_qps, "unit": "queries/s",
                                             "note": "score + flatnonzero/argpartition top-k, informational"},
                         "cold": cold},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(args, queries_per_step):
    return {"workload": "10M-doc synthetic MSMARCO, single-term BM25, top-%d (BASELINE configs[1])" % args.k,
            "n_docs": args.docs, "queries_per_step": queries_per_step, "k": args.k,
            "corpus": "searcharray_b200.synth seed 20260924, doc_lens~floor(clip(lognormal(3.9,.45),8,400)), "
                      "1024 DISTINCT query terms over df/N in {3e-1..1e-4}, every term once per step",
            "sharding": "contiguous doc-id ranges, one process per GPU",
            "cache": "inputs larger than L2: every step streams its own posting lists (8 GB at 10M docs) and "
                     "queries_per_step dense float32[N] vectors"}


# --------------------------------------------------------------------------- our arm
class Ours:
    """Thin harness around one shard's sa_index handle and the batch API."""

    def __init__(self, args, rank, world):
        from searcharray_b200 import _lib
        from searcharray_b200.postings import DeviceIndex
        self._lib = _lib
        self.L = _lib.lib()
        self.args, self.rank, self.world = args, rank, world
        self.local_rank = int(os.environ.get("LOCAL_RANK", rank))
        self.spec, self.host, self.lo, self.hi, self.avgdl = build_corpus(args.docs, rank, world)
        t0 = time.time()
        self.dev = DeviceIndex(self.host, device=self.local_rank, doc_base=self.lo)
        log(f"rank {rank}: upload {time.time() - t0:.1f}s")
        self.h = self.dev.handle
        self.ms = ctypes.c_double(0)
        self.n_over = ctypes.c_uint32(0)
        dbg("uploaded")
        if world > 1:
            self._init_comm()
        dbg("comm ready")
        L, h = self.L, self.h
        df = np.zeros(self.host.n_terms, dtype=np.uint64)
        tmp = ctypes.c_uint64(0)
        for t in range(self.host.n_terms):
            _lib.check(L.sa_docfreq(h, t, ctypes.byref(tmp)))
            df[t] = tmp.value
        self.df_local = df.copy()
        if world > 1:
            _lib.check(L.sa_comm_allreduce_sum_u64(h, _lib.p_u64(df), len(df)))
        self.df = df                       # GLOBAL document frequencies (idf must not depend on sharding)
        dbg("global df done")

    def _init_comm(self):
        _lib, L, h, rank, world = self._lib, self.L, self.h, self.rank, self.world
        # NCCL_DEBUG=VERSION/WARN print a banner on STDOUT, which would break the one-JSON-line contract
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION", "WARN"):
            os.environ.pop("NCCL_DEBUG", None)
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/sa_b200_nccl_%h_%p.log")
        # one node, NVLink/NVSwitch between the GPUs: the bootstrap sockets stay on loopback and NCCL does not probe
        # InfiniBand / network plugins (probing them made ncclCommInitRank take 18 s here, and once never return)
        os.environ.setdefault("NCCL_SOCKET_IFNAME", "lo")
        os.environ.setdefault("NCCL_IB_DISABLE", "1")
        # Rendezvous for the NCCL unique id without any framework: all ranks of one launch share a
        # node (contract: --nnodes=1) and a parent (the torchrun agent), so rank 0 publishes the id
        # in a file keyed by MASTER_PORT + parent pid and the others poll for it.
        key = f"/tmp/sa_b200_uid_{os.environ.get('MASTER_PORT', '0')}_{os.getppid()}.bin"
        uid = (ctypes.c_char * 128)()
        if rank == 0:
            _lib.check(L.sa_comm_unique_id(uid))
            with open(key + ".tmp", "wb") as f:
                f.write(bytes(uid))
            os.replace(key + ".tmp", key)
        else:
            t_wait = time.time()
            while not os.path.exists(key):
                if time.time() - t_wait > 900:
                    raise RuntimeError("timed out waiting for rank 0's NCCL id")
                time.sleep(0.05)
            with open(key, "rb") as f:
                uid = (ctypes.c_char * 128).from_buffer_copy(f.read(128))
        _lib.check(L.sa_comm_init(h, uid, rank, world))
        _lib.check(L.sa_comm_barrier(h))
        if rank == 0:
            os.remove(key)

    def barrier(self):
        if self.world > 1:
            self._lib.check(self.L.sa_comm_barrier(self.h))

    def max_over_ranks(self, x):
        v = ctypes.c_double(x)
        if self.world > 1:
            self._lib.check(self.L.sa_comm_allreduce_max(self.h, ctypes.byref(v)))
        return v.value

    # ---- the batch API
    def upload(self, terms, starts, idf, slop, k):
        _lib = self._lib
        _lib.check(self.L.sa_batch_upload(self.h, _lib.p_u32(terms), _lib.p_u32(starts), _lib.p_f32(idf),
                                          len(starts) - 1, slop, float(self.avgdl), K1, B, k))

    def execute(self):
        self._lib.check(self.L.sa_batch_execute_allgather(self.h) if self.world > 1 else self.L.sa_batch_execute(self.h))

    def download(self, docs, scores):
        _lib = self._lib
        fn = self.L.sa_batch_download_allgather if self.world > 1 else self.L.sa_batch_download
        _lib.check(fn(self.h, _lib.p_u32(docs), _lib.p_f32(scores), ctypes.byref(self.n_over)))
        return self.n_over.value

    def timed_executes(self, steps):
        """K x execute between CUDA events on the library's stream; max over ranks, in ms."""
        _lib, L, h = self._lib, self.L, self.h
        self.barrier()
        _lib.check(L.sa_timer_start(h))
        for _ in range(steps):
            self.execute()
        _lib.check(L.sa_timer_stop(h, ctypes.byref(self.ms)))
        self.barrier()
        return self.max_over_ranks(self.ms.value)

    def stats(self):
        st = self._lib.SaStats()
        self._lib.check(self.L.sa_stats_get(self.h, ctypes.byref(st)))
        return st

    def profiled(self, steps):
        """term / phrase kernel ms per step from per-launch CUDA events (async, resolved at the end)."""
        _lib, L, h = self._lib, self.L, self.h
        _lib.check(L.sa_set_profiling(h, 1))
        _lib.check(L.sa_stats_reset(h))
        for _ in range(steps):
            self.execute()
        st = self.stats()
        _lib.check(L.sa_set_profiling(h, 0))
        return st


def peak_hbm():
    peak, src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak, src = float(mp["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        pass
    return peak, src


def committed_traffic(kernel, cfg):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture of this very
    workload (it cannot be measured live); None for any other configuration."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))
        for ent in tj.get(kernel, []):
            if ent["config"] == cfg:
                return float(ent["dram_bytes_read_per_launch"] + ent["dram_bytes_write_per_launch"]), ent["source"]
    except Exception:
        pass
    return None, None


def oracle_topk_term(full, avgdl, idf, term_id, k):
    """The oracle's top-k keys for one term query: sparse tf (popcount64_reduce) -> BM25 on the
    matching docs (bm25.pyx:20-25, bit-identical to scoring all N: tf == 0 scores +0.0) -> top-k."""
    from oracle import ops as oops, search as osearch
    from searcharray_b200.shard import shard_topk_keys, unpack_keys
    ids, tfs = osearch.termfreqs_sparse(full.term_words(term_id))
    sc = tfs.copy()
    oops.bm25_score(sc, full.doc_lens[ids.astype(np.int64)], avgdl, float(idf), K1, B)
    return unpack_keys(shard_topk_keys(ids, sc, k))


def topk_of_dense(dense, k):
    d, s = cpu_topk(dense, k)
    docs = np.full(k, 0xFFFFFFFF, dtype=np.uint32)
    scores = np.zeros(k, dtype=np.float32)
    docs[:len(d)] = d
    scores[:len(s)] = s
    return docs, scores


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, docs, scores):
    """Writes the global top-k of the last timed step as <out_dir>/topk_docs.npy (float64 doc ids, exact;
    0xFFFFFFFF = no doc) and topk_scores.npy (float32), one row per query, so that two builds can be compared
    output for output.  Above 64 MB in all, a fixed seeded sample of the rows is written, with its row numbers
    in topk_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    rows = np.arange(docs.shape[0])
    max_rows = (DUMP_LIMIT_BYTES - 4096) // (docs.shape[1] * (8 + 4) + 8)      # 4 KB for the .npy headers
    if len(rows) > max_rows:
        rows = np.sort(np.random.default_rng(0).choice(len(rows), max_rows, replace=False))
        np.save(os.path.join(out_dir, "topk_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "topk_docs.npy"), docs[rows].astype(np.float64))
    np.save(os.path.join(out_dir, "topk_scores.npy"), scores[rows].astype(np.float32))


def bench_ours(args, rank, world):
    from searcharray_b200 import synth
    o = Ours(args, rank, world)
    _lib, L, h, host, spec, avgdl, df = o._lib, o.L, o.h, o.host, o.spec, o.avgdl, o.df
    names, term_ids = make_queries(spec, args.queries)
    idf = idf_of(args.docs, df[term_ids])
    starts = np.arange(len(term_ids) + 1, dtype=np.uint32)
    Q, k = len(term_ids), args.k
    out_docs = np.empty((Q, k), dtype=np.uint32)
    out_scores = np.empty((Q, k), dtype=np.float32)

    def e2e_step():
        o.upload(term_ids, starts, idf, 0, k)
        o.execute()
        return o.download(out_docs, out_scores)

    # ---- warm-up (>= 3 full steps); the clock sampler (nvidia-smi -lms) starts here so that it is
    #      already delivering samples when the timed region begins
    clocks = ClockSampler(o.local_rank)
    clocks.start()
    overflow = 0
    for _ in range(max(args.warmup, 3)):
        overflow += e2e_step()
        dbg("warm-up step done")

    # ---- value: device-resident, K x execute between CUDA events on the library stream
    o.upload(term_ids, starts, idf, 0, k)
    _lib.check(L.sa_stats_reset(h))
    t_timed = time.time()
    dev_ms = o.timed_executes(args.steps)
    launches_value = int(o.stats().total_launches)
    o.download(out_docs, out_scores)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out_docs, out_scores)
    value = args.steps * Q / (dev_ms / 1e3)
    dbg("device-timed steps done")

    # ---- e2e: host buffers in, top-k out, every step
    o.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        overflow += e2e_step()
    o.barrier()
    e2e_s = o.max_over_ranks(time.perf_counter() - t0)
    e2e = args.steps * Q / e2e_s
    t_timed_end = time.time()
    # clocks: samples taken during the two timed regions (device-timed steps + e2e steps).  When those
    # are shorter than a few sampling periods (many GPUs, small shards) the same step is repeated,
    # untimed, for ~0.4 s so that the clocks under this load are still observed.
    clock_note = "sampled during the timed regions"
    if clocks.count_since(t_timed) < 4:
        n_extra = int(min(2000, max(1, 0.4 / max(dev_ms / 1e3 / args.steps, 1e-5))))
        for _ in range(n_extra):
            o.execute()
        o.barrier()
        o.download(out_docs, out_scores)
        t_timed_end = time.time()
        clock_note = f"timed regions too short to sample: + {n_extra} untimed repeats of the same step"
    clk = clocks.stop(t_timed)          # (nvidia-smi's piped output arrives in bursts: no upper time bound)
    clk["note"] = clock_note
    h2d = int(term_ids.nbytes + starts.nbytes + idf.nbytes + Q * 32)     # + TermQuery descriptors
    d2h = int(Q * k * 8 + Q * 4)

    # ---- roofline of the dominant kernel (per-launch CUDA events, async)
    W = host.term_lengths[term_ids].astype(np.float64)
    dfl = o.df_local.astype(np.float64)
    # per query, this shard (SURVEY 8d).  Lists with a tile directory are scanned through the tf table the index
    # builds at upload -- one 4-byte (doc, tf) record per matching doc instead of the 8-byte posting words -- so
    # their posting term is 4*df ("its actual record size"); short lists are still scanned as words (8*W).
    n_tiles = (host.n_docs + 8191) // 8192
    has_table = (W >= max(1024, n_tiles // 2)) & (os.environ.get("SA_NO_TF_TABLE", "0") in ("", "0"))
    post_bytes = np.where(has_table, 4.0 * dfl[term_ids], 8.0 * W)
    alg_q = post_bytes + 4.0 * dfl[term_ids] + 4.0 * host.n_docs
    prof_steps = min(args.steps, 5)
    st = o.profiled(prof_steps)
    term_ms = st.term_kernel_ms / prof_steps
    launches_per_step = st.term_kernel_launches / prof_steps
    achieved = float(alg_q.sum()) / (term_ms / 1e3) / 1e9
    peak, peak_src = peak_hbm()
    traffic, traffic_src = committed_traffic("term_tile_kernel", {"n_docs": args.docs, "queries_per_step": Q, "n_gpus": world})
    roofline = {"bound": "hbm", "kernel": "term_tile_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "frac_of_nominal_8TBs": achieved / 8000.0,      # SURVEY 8d: both denominators
                "algorithmic_bytes_per_launch": float(alg_q.sum()) / launches_per_step,
                "algorithmic_bytes": "postings + 4*df (norms) + 4*N (dense row) per query (SURVEY 8d), summed over the "
                                     "launch's queries; postings = 4*df for lists scanned through the upload-time "
                                     "(doc, tf) record table, 8*W for short lists scanned as words",
                "tf_table_queries": int(np.count_nonzero(has_table)),
                "avg_launch_ms": term_ms / launches_per_step, "launches_per_step": launches_per_step,
                "topk_select_ms_per_step": st.topk_kernel_ms / prof_steps,
                "kernel_share_of_step": term_ms / (dev_ms / args.steps)}
    # per-df-bucket fractions: the same kernel over the queries of ONE bucket at a time
    buckets = []
    qb = np.asarray([spec.terms[t][2] for t in term_ids])
    for bi, p in enumerate(synth.DF_BUCKETS):
        sel = np.flatnonzero(qb == bi)
        if len(sel) == 0:
            continue
        o.upload(np.ascontiguousarray(term_ids[sel]), np.arange(len(sel) + 1, dtype=np.uint32),
                 np.ascontiguousarray(idf[sel]), 0, k)
        for _ in range(2):
            o.execute()
        stb = o.profiled(3)
        ms_b = stb.term_kernel_ms / 3
        b_docs = np.empty((len(sel), k), dtype=np.uint32)
        b_scores = np.empty((len(sel), k), dtype=np.float32)
        buckets.append({"df_over_n": p, "queries": int(len(sel)), "us_per_query": 1e3 * ms_b / len(sel),
                        "topk_overflow_reruns": int(o.download(b_docs, b_scores)),
                        "achieved": float(alg_q[sel].sum()) / (ms_b / 1e3) / 1e9,
                        "frac": float(alg_q[sel].sum()) / (ms_b / 1e3) / 1e9 / peak})
    roofline["by_df_bucket"] = buckets
    dbg("buckets done")
    o.upload(term_ids, starts, idf, 0, k)

    # ---- verify: GPU top-k (docs AND score bits) against the oracle, rank 0 holds the FULL corpus
    verify = None
    n_verify = args.verify if args.verify >= 0 else (48 if world == 1 else 16)
    full = None
    if n_verify:
        o.execute()
        o.download(out_docs, out_scores)
        if rank == 0:
            full = host if world == 1 else synth.generate_shard(spec, 0, 1)[0]
            step = max(1, Q // n_verify)
            checked, bad = 0, 0
            for qi in list(range(0, Q, step))[:n_verify]:
                wd, ws = oracle_topk_term(full, avgdl, idf[qi], int(term_ids[qi]), k)
                checked += 1
                if not (np.array_equal(wd, out_docs[qi]) and
                        np.array_equal(ws.view(np.uint32), out_scores[qi].view(np.uint32))):
                    bad += 1
            verify = {"term": {"queries_checked": checked, "mismatches": bad,
                               "what": "global top-%d doc ids and score bits vs the CPU oracle" % k}}
            log("verify term:", verify["term"])

    dbg("term verify done")
    # ---- phrase workloads (BASELINE configs[2] and [3]) as extra blocks
    phrase = None
    bigram = None
    cpu_arm = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_arm = CpuArm(spec, host, avgdl, args.docs)

    def phrase_batch(queries, slop):
        ids = [[spec.term_index[t] for t in ph] for ph in queries]
        p_terms = np.asarray([t for ph in ids for t in ph], dtype=np.uint32)
        p_starts = np.concatenate(([0], np.cumsum([len(ph) for ph in ids]))).astype(np.uint32)
        p_idf = np.asarray([phrase_idf(args.docs, df, ph) for ph in ids], dtype=np.float32)
        return ids, p_terms, p_starts, p_idf

    def phrase_block(queries, slop, label, with_roofline):
        """One batched pass family of phrase queries with `slop`: device-timed steps, the same steps
        end to end (upload + execute + top-k download), B_phrase roofline, parity sample."""
        ids, p_terms, p_starts, p_idf = phrase_batch(queries, slop)
        PQ = len(queries)
        dbg("phrase block start:", label[:48], "slop", slop, "queries", PQ)
        p_docs = np.empty((PQ, k), dtype=np.uint32)
        p_scores = np.empty((PQ, k), dtype=np.float32)
        p_redo = 0
        for _ in range(3):
            o.upload(p_terms, p_starts, p_idf, slop, k); o.execute(); p_redo += o.download(p_docs, p_scores)
        dbg("  warm-up done, repairs", p_redo)
        o.upload(p_terms, p_starts, p_idf, slop, k)
        p_steps = args.steps
        p_ms = o.timed_executes(p_steps)
        dbg("  timed done")
        _lib.check(L.sa_stats_reset(h))
        o.execute()
        o.download(p_docs, p_scores)
        st1 = o.stats()
        o.barrier()
        t0 = time.perf_counter()
        for _ in range(p_steps):
            o.upload(p_terms, p_starts, p_idf, slop, k); o.execute(); p_redo += o.download(p_docs, p_scores)
        o.barrier()
        p_e2e_s = o.max_over_ranks(time.perf_counter() - t0)
        Wp = np.asarray([float(np.sum(host.term_lengths[ph])) for ph in ids])
        blk = {"workload": label, "queries_per_step": PQ, "distinct_queries": len({tuple(q) for q in queries}),
               "value": p_steps * PQ / (p_ms / 1e3), "unit": "queries/s", "ms_per_step": p_ms / p_steps,
               "e2e": {"value": p_steps * PQ / p_e2e_s, "unit": "queries/s"}, "repairs": int(p_redo),
               "queries_with_matches": int(np.sum(p_docs[:, 0] != 0xFFFFFFFF)),
               "mean_words_per_query_this_shard": float(np.mean(Wp)),
               "min_list_words_mean": float(np.mean([np.min(host.term_lengths[ph]) for ph in ids]))}
        if with_roofline:
            stp = o.profiled(min(p_steps, 3))
            k_ms = stp.phrase_kernel_ms / min(p_steps, 3)
            alg = 8.0 * float(Wp.sum()) + 16.0 * st1.phrase_cont_words + 4.0 * host.n_docs * PQ + 4.0 * st1.phrase_matched_docs
            tr, tr_src = committed_traffic("phrase_kernel", {"n_docs": args.docs, "queries_per_step": PQ, "n_gpus": world,
                                                            "workload": label})
            blk["roofline"] = {"bound": "hbm", "kernel": "phrase kernels (slop 0)", "achieved": alg / (k_ms / 1e3) / 1e9,
                               "peak": peak, "unit": "GB/s", "frac": alg / (k_ms / 1e3) / 1e9 / peak,
                               "traffic": tr, "traffic_source": tr_src,
                               "algorithmic_bytes": "B_phrase = 8*sum(W) + 16*sum(C_s) + 4*N + 4*M (SURVEY 8d)",
                               "algorithmic_bytes_per_step": alg, "sum_W_words": float(Wp.sum()),
                               "sum_C_words": int(st1.phrase_cont_words), "matched_docs": int(st1.phrase_matched_docs),
                               "kernel_ms_per_step": k_ms, "kernel_share_of_step": k_ms / (p_ms / p_steps),
                               "note": "lists that a search skips are still credited: a fraction above 1 means the "
                                       "kernel read less than B_phrase"}
        # parity sample against the CPU arm's dense vector (score bits and doc ids of the top-k)
        if cpu_arm is not None and n_verify:
            nck = min(args.verify_phrases, PQ)
            stepq = max(1, PQ // nck)
            bad, t_cpu = 0, 0.0
            for qi in list(range(0, PQ, stepq))[:nck]:
                t0 = time.perf_counter()
                dense = cpu_arm.score_phrase(ids[qi], slop=slop)
                t_cpu += time.perf_counter() - t0
                wd, ws = topk_of_dense(dense, k)
                if not (np.array_equal(wd, p_docs[qi]) and np.array_equal(ws.view(np.uint32), p_scores[qi].view(np.uint32))):
                    bad += 1
            blk["verify"] = {"queries_checked": nck, "mismatches": bad,
                             "what": "top-%d doc ids and score bits vs the CPU %s's dense .score()" % (k, cpu_arm.kind)}
            blk["cpu_baseline"] = {"kind": cpu_arm.kind, "cores": 1, "value": nck / t_cpu, "unit": "queries/s",
                                   "sample": f"{nck} of the step's queries, SearchArray.score(phrase, slop={slop}), one thread"}
            log(label, "verify:", blk["verify"], "cpu q/s: %.1f" % (nck / t_cpu))
        return blk

    if args.phrase_queries > 0:
        pq_all = synth.phrase_queries(spec, args.phrase_queries)
        kinds = synth.phrase_kinds(spec, pq_all)
        phrase = phrase_block(pq_all, 0, "4-term phrase, slop 0 (BASELINE configs[2]): 3/4 with one rare term "
                              "(df/N <= 1e-3), 1/4 'hard' (all df/N >= 1e-2), planted + natural matches, top-%d" % k, True)
        rare_q = [q for q, kd in zip(pq_all, kinds) if kd == "rare"]
        hard_q = [q for q, kd in zip(pq_all, kinds) if kd == "hard"]
        if rare_q and hard_q:
            phrase["rare_only"] = phrase_block(rare_q, 0, "4-term phrase, slop 0, rare-term stratum", True)
            phrase["hard_only"] = phrase_block(hard_q, 0, "4-term phrase, slop 0, hard stratum (all df/N >= 1e-2)", True)
        if args.slop_queries > 0:
            phrase["slop2"] = phrase_block(pq_all[:args.slop_queries], 2,
                                           "4-term phrase, slop 2 (BASELINE configs[3]), same batched top-%d API" % k, False)
            if rare_q and hard_q and args.slop_queries >= 64:
                phrase["slop2_rare"] = phrase_block(rare_q[:args.slop_queries], 2, "4-term phrase, slop 2, rare-term stratum", False)
                phrase["slop2_hard"] = phrase_block(hard_q[:args.slop_queries], 2, "4-term phrase, slop 2, hard stratum", False)
        bq = synth.bigram_queries(spec, args.bigram_queries)
        if bq:
            bigram = phrase_block(bq, 0, "bigram common (df/N 3e-1) x mid (df/N 3e-2), slop 0 (BASELINE.md's 4.5M x 0.45M-word "
                                  "case), top-%d" % k, True)
        # slop = 2 through the per-query C-ABI call (the .score(..., slop=2) drop-in, dense vector to the host)
        if rank == 0 and world == 1 and args.slop_queries > 0:
            from searcharray_b200.postings import _pool
            ids, p_terms, p_starts, p_idf = phrase_batch(pq_all[:16], 2)
            out = _pool.empty_f32(host.n_docs)
            _lib.check(L.sa_set_profiling(h, 1))
            _lib.check(L.sa_stats_reset(h))
            matched, dt = 0, 0.0
            for i, ph in enumerate(ids):
                tids = np.ascontiguousarray(ph, dtype=np.uint32)
                t0 = time.perf_counter()
                _lib.check(L.sa_score_phrase(h, _lib.p_u32(tids), len(tids), 2, float(p_idf[i]), float(avgdl), K1, B, 0,
                                             _lib.ALL_BITS, _lib.p_f32(out)))
                dt += time.perf_counter() - t0
                matched += int(np.count_nonzero(out))
            stq = o.stats()
            _lib.check(L.sa_set_profiling(h, 0))
            phrase["slop2_dense"] = {"workload": "4-term phrase, slop 2, sa_score_phrase per query (the .score() drop-in), "
                                                 "dense float32[N] to the host", "queries": len(ids),
                                     "e2e": {"value": len(ids) / dt, "unit": "queries/s"},
                                     "kernel_ms_per_query": stq.phrase_kernel_ms / len(ids),
                                     "mean_matching_docs": matched / len(ids)}
        o.upload(term_ids, starts, idf, 0, k)          # restore the term batch for the sections below

    dbg("phrase blocks done")
    # ---- edismax (the shape of BASELINE configs[4], on this run's corpus size): two fields, mixed
    #      2-5 term queries, qf + pf + pf2 + pf3, mm=2, tie=0.3 (reference test_msmarco.py:436-443)
    edis = None
    if args.edismax_queries > 0:
        edis = edismax_block(args, o, cpu_arm)
        o.upload(term_ids, starts, idf, 0, k)

    # ---- e2e_dense: the literal .score() drop-in, dense float32[N] to the host per query
    e2e_dense = None
    if rank == 0 and world == 1:
        from searcharray_b200.postings import _pool
        out = _pool.empty_f32(host.n_docs)
        nd = min(Q, 96)
        for i in range(3):
            _lib.check(L.sa_score_term(h, int(term_ids[i]), float(idf[i]), float(avgdl), K1, B, 0, _lib.ALL_BITS,
                                       _lib.p_f32(out)))
        t0 = time.perf_counter()
        for i in range(nd):
            _lib.check(L.sa_score_term(h, int(term_ids[i]), float(idf[i]), float(avgdl), K1, B, 0, _lib.ALL_BITS,
                                       _lib.p_f32(out)))
        dt = time.perf_counter() - t0
        e2e_dense = {"value": nd / dt, "unit": "queries/s", "d2h_bytes_per_query": int(host.n_docs * 4),
                     "note": "SearchArray.score drop-in: one sa_score_term call per query, pinned result vector"}
        # dense parity at the BASELINE size: one term per df bucket, the whole float32[N] bit for bit
        if cpu_arm is not None and n_verify:
            bad = 0
            picks = [int(np.flatnonzero(qb == bi)[0]) for bi in range(len(synth.DF_BUCKETS)) if np.any(qb == bi)]
            for qi in picks:
                _lib.check(L.sa_score_term(h, int(term_ids[qi]), float(idf[qi]), float(avgdl), K1, B, 0, _lib.ALL_BITS,
                                           _lib.p_f32(out)))
                want = cpu_arm.score_term(int(term_ids[qi]))
                if not np.array_equal(out.view(np.uint32), want.view(np.uint32)):
                    bad += 1
            verify = verify or {}
            verify["dense"] = {"vectors_checked": len(picks), "mismatches": bad,
                               "what": "sa_score_term float32[N] bit-for-bit vs the CPU %s's .score(), one term per df bucket"
                                       % cpu_arm.kind}
            log("verify dense:", verify["dense"])

    # ---- cpu_baseline (rank 0, N=1): the reference's .score() on the host cores, bounded sample
    cpu = None
    if cpu_arm is not None:
        cores = os.cpu_count() or 1
        sample = term_ids[:min(Q, args.ref_sample)]
        cpu_arm.warm(sample, threads=min(cores, 32))
        threads, _ = best_thread_count(cpu_arm.score_term, sample, cores)
        tt, n = 0.0, 0
        while tt < 10.0 and n < 8:
            tt += run_cpu_sample(cpu_arm.score_term, sample, threads)
            n += 1
        one_thread = len(sample[:32]) / run_cpu_sample(cpu_arm.score_term, sample[:32], 1)
        tk = sample[:24]
        topk_qps = len(tk) / run_cpu_sample(lambda q: cpu_topk(cpu_arm.score_term(q), k), tk, min(threads, 8))
        cpu = {"value": n * len(sample) / tt, "unit": "queries/s", "cores": threads, "host_cores": cores,
               "kind": cpu_arm.kind,
               "sample": f"{n} x {len(sample)} of the step's queries, stock SearchArray.score (dense float32[N], no top-k), "
                         f"ThreadPool({threads}) = fastest of the probed pool widths, warm tf/df caches",
               "one_thread": {"value": one_thread, "unit": "queries/s"},
               "score_plus_topk": {"value": topk_qps, "unit": "queries/s",
                                   "note": "score + flatnonzero/argpartition top-k, informational"}}
        try:
            cpu["cold"] = cold_cpu_qps(cpu_arm, sample)
        except Exception as e:                      # informational; never fail the run for it
            cpu["cold"] = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": "queries/sec (single-term BM25 + top-k) on 10M-doc synthetic MSMARCO",
            "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, Q),
            "clocks": clk,
            "e2e": {"value": e2e, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches_value,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "e2e_dense": e2e_dense,
            "phrase": phrase,
            "bigram": bigram,
            "edismax": edis,
            "topk_overflow_reruns": int(overflow),
            "verify": verify,
        }
        print(json.dumps(line), flush=True)
    o.dev.close()


def edismax_block(args, o, cpu_arm):
    import pandas as pd
    from searcharray_b200 import SearchArray, solr, synth
    from searcharray_b200.shard import ShardComm
    _lib, L = o._lib, o.L
    k, rank, world = args.k, o.rank, o.world
    t0 = time.time()
    tspec, thost, _, _, t_avgdl = build_corpus(args.docs, rank, world, field="title")
    comm = ShardComm(o.h, rank, world)
    body = SearchArray.from_host_index(o.host, device=o.local_rank, doc_base=o.lo, corpus_size=args.docs,
                                       avg_doc_length=o.avgdl, global_df=o.df, comm=comm)
    body._shared["dev"] = o.dev                      # the body shard is already in HBM
    title = SearchArray.from_host_index(thost, device=o.local_rank, doc_base=o.lo, corpus_size=args.docs,
                                        avg_doc_length=t_avgdl, comm=comm)
    tdev = title._device()
    tdf = np.zeros(thost.n_terms, dtype=np.uint64)
    tmp = ctypes.c_uint64(0)
    for t in range(thost.n_terms):
        _lib.check(L.sa_docfreq(tdev.handle, t, ctypes.byref(tmp)))
        tdf[t] = tmp.value
    title.global_df = comm.sum_u64(tdf)
    frame = pd.DataFrame({"title": title, "body": body})
    log(f"edismax: title field {thost.words.nbytes / 1e6:.0f} MB of postings, avgdl={t_avgdl}, "
        f"set-up {time.time() - t0:.1f}s")
    eq = synth.edismax_queries(o.spec, args.edismax_queries)
    ekw = dict(qf=["title^1.0", "body^0.5"], pf=["title", "body"], pf2=["title", "body"], pf3=["title", "body"],
               mm=2, tie=0.3)
    for qtext in eq[:3]:
        solr.edismax_topk(frame, qtext, k=k, **ekw)
    o.barrier()
    solr._TIMING = {}
    t0 = time.perf_counter()
    hits = 0
    for qtext in eq:
        d_, s_ = solr.edismax_topk(frame, qtext, k=k, **ekw)
        hits += int(d_[0] != 0xFFFFFFFF)
    o.barrier()
    e_s = o.max_over_ranks(time.perf_counter() - t0)
    call_ms = {kk: 1e3 * vv / len(eq) for kk, vv in solr._TIMING.items()}
    solr._TIMING = None
    edis = {"workload": "two-field edismax (title^1.0 body^0.5, pf/pf2/pf3 on both fields as test_msmarco.py:436-443, mm=2, "
                        "tie=0.3), mixed 2-5 term queries, exact float64 top-%d" % k,
            "queries": len(eq), "e2e": {"value": len(eq) / e_s, "unit": "queries/s"},
            "ms_per_query": 1e3 * e_s / len(eq), "queries_with_hits": hits,
            "ms_per_query_by_call": call_ms}
    if cpu_arm is not None:
        from oracle import search as osearch, solr as osolr
        ofields = {}
        for name, hidx, adl in (("title", thost, t_avgdl), ("body", o.host, o.avgdl)):
            oi = osearch.OracleIndex({t: hidx.term_words(t) for t in range(hidx.n_terms)}, hidx.doc_lens,
                                     avg_doc_length=adl, corpus_size=args.docs, cache=True)
            ofields[name] = osolr.OracleField(oi, hidx.term_dict.term_to_ids)
        nq = min(args.verify_edismax, len(eq))
        t_cpu, bad = 0.0, 0
        for qtext in eq[:nq]:
            t0 = time.perf_counter()
            want = osolr.edismax(ofields, qtext, **ekw)
            t_cpu += time.perf_counter() - t0
            d_, s_ = solr.edismax_topk(frame, qtext, k=k, **ekw)
            order = np.lexsort((np.arange(len(want)), -want))[:k]
            order = order[want[order] > 0]
            if not (np.array_equal(d_[:len(order)], order.astype(np.uint32)) and
                    np.allclose(s_[:len(order)], want[order], rtol=1e-5, atol=0)):
                bad += 1
        edis["cpu_baseline"] = {"kind": "port", "cores": 1, "value": nq / t_cpu, "unit": "queries/s",
                                "sample": f"{nq} of the queries, oracle port of solr.py (oracle/solr.py)"}
        edis["verify"] = {"queries_checked": nq, "mismatches": bad,
                          "what": "top-%d docs exact, float64 scores within 1e-5 vs oracle/solr.py" % k}
    del frame, title, tdev
    return edis


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--docs", type=int, default=10_000_000)
    ap.add_argument("--queries", type=int, default=1024)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--ref-sample", type=int, default=192)
    ap.add_argument("--ref-budget", type=float, default=150.0,
                    help="reference arm: target seconds for all --steps + --warmup passes (bounds the per-step sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--phrase-queries", type=int, default=256)
    ap.add_argument("--slop-queries", type=int, default=256)
    ap.add_argument("--bigram-queries", type=int, default=32)
    ap.add_argument("--edismax-queries", type=int, default=48)
    ap.add_argument("--verify", type=int, default=-1,
                    help="term queries whose global top-k (docs + score bits) is checked against the CPU oracle "
                         "(default 48 at 1 GPU, 16 sharded -- rank 0 then re-generates the FULL corpus; 0 = off)")
    ap.add_argument("--verify-phrases", type=int, default=12)
    ap.add_argument("--verify-edismax", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the top-k doc ids and scores of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        bench_reference(args, rank, world)
    else:
        bench_ours(args, rank, world)


if __name__ == "__main__":
    main()
