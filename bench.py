#!/usr/bin/env python
"""bench.py -- throughput of the alignment hot path on B200 (metric of BASELINE.json: GCUPS = sum(qLen*tLen)/1e9/s).

Default workload (N=1) = BASELINE config[1]: ungapped prefilter, L~350 protein queries against a 1M-sequence synthetic
target DB.  One "step" = one batch of queries scanned against the whole resident DB (the reference's own unit of work is
one query per Marv::scan / runFilterOnCpu pass; the DB is loaded once, as Marv::loadDb / gpuserver do).
  value     : GCUPS with the query profiles already staged in HBM (b200_scan_job_* ; CUDA events on the library's stream)
  e2e       : GCUPS through the public C-ABI call with HOST buffers (b200_ungapped_scan: H2D profiles, kernels, top-k, D2H hits)
  secondary : BASELINE config[2] (gapped SW rescoring, L 50-2000, gap 11/1) measured the same two ways
  roofline  : integer-pipe roofline of the dominant kernel (SURVEY.md 8d: this path is int-pipe bound, not HBM bound; the
              HBM figures are reported next to it to show that), peak = DPX issue rate measured live by
              profiles/microbench/int_pipe_rate on this GPU
  cpu_baseline : the reference's own AVX2 code (oracle/_ref, built in place from /root/reference) on the host cores, bounded sample

`--impl reference` times the reference's CPU implementation (same metric/config) instead.
N>1 (torchrun): queries are sharded across ranks (DB replicated, no data-path collective), per-step top-k hit lists are
gathered to every rank with one NCCL all_gather; weak scaling (fixed queries per GPU per step).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "GCUPS"
SCAN_OPS_PER_CELL = 0.75   # DESIGN.md: per 2 cells 1 VIADDMNMX.S16x2.RELU + 0.5 VIMNMX3.S16x2
SW32_OPS_PER_CELL = 6.0    # DESIGN.md: sw32 kernel, 6 int instructions per cell (int32, one cell per instruction)
SW16_OPS_PER_CELL = 3.25   # DESIGN.md: sw16 kernel, 6.5 DPX/PRMT instructions per packed register = 2 cells


def load_matrix():
    d = np.load(os.path.join(ROOT, "tests", "golden", "blosum62.npz"))
    return d["mat"], d["pback"]


def make_scan_workload(rank, db_seqs, queries_per_step, n_steps_distinct):
    """config[1]: DB identical on every rank (seed 2), queries rank-specific (seed 1000+rank)."""
    from mmseqs2_b200 import synth
    mat, pb = load_matrix()
    bg = synth.background(pb)
    rng_db = np.random.default_rng(2)
    res, off = synth.random_seqs(rng_db, db_seqs, bg, mean=300.0, sigma=0.6, lo=30, hi=5000)
    rng_q = np.random.default_rng(1000 + rank)
    nq = queries_per_step * n_steps_distinct
    qres, qoff = synth.random_seqs(rng_q, nq, bg, mean=350.0, sigma=35.0, lo=200, hi=500, normal=True)
    queries = synth.split(qres, qoff)
    rng_p = np.random.default_rng(3)
    synth.plant_homologs(rng_p, res, off, queries[:min(len(queries), 64)], bg, frac=min(0.01, 2000.0 / db_seqs))
    return res, off, queries


def make_sw_workload(n_queries, targets_per_query):
    """config[2]: (query,target) pairs -- prefilter-hit lists of n_queries queries --, lengths log-uniform in [50,2000], half of
    every list random sequences, half homologs of the query at 20-90 % identity with indels, so byte and word modes are both
    exercised.  n_queries x targets_per_query = the number of pairs (BASELINE: 1 M)."""
    from mmseqs2_b200 import synth
    mat, pb = load_matrix()
    bg = synth.background(pb)
    cdf = np.cumsum(bg)
    rng = np.random.default_rng(77)
    n_hom = targets_per_query // 2
    n_rand = targets_per_query - n_hom
    # one pool of random targets shared by all lists (drawn without replacement per query); homologs generated per query
    pool_n = max(4 * n_rand, 4096)
    pool_len = np.exp(rng.uniform(np.log(50), np.log(2000), pool_n)).astype(np.int64)
    chunks = [np.minimum(np.searchsorted(cdf, rng.random(int(pool_len.sum())), side="right"), 19).astype(np.uint8)]
    lens = [pool_len]
    queries, pairs = [], []
    n_targets = pool_n
    gen = None
    try:   # homolog generation on the GPU when there is one (data plumbing; the numpy path produces the same kind of data, slower)
        import torch
        if torch.cuda.is_available():
            gen = torch.Generator(device="cuda")
            gen.manual_seed(77)
    except Exception:
        gen = None
    for qi in range(n_queries):
        L = int(np.exp(rng.uniform(np.log(50), np.log(2000))))
        q = np.minimum(np.searchsorted(cdf, rng.random(L), side="right"), 19).astype(np.uint8)
        queries.append(q)
        ids = np.empty(targets_per_query, np.int64)
        ids[:n_rand] = rng.choice(pool_n, n_rand, replace=False)
        if n_hom:
            if gen is not None:
                hd, hl = synth.mutate_many_torch(gen, q, n_hom, 0.2, 0.9, 0.02)
                hd, hl = hd.cpu().numpy(), hl.cpu().numpy()
            else:
                hd, hl = synth.mutate_many(rng, q, n_hom, bg, 0.2, 0.9, 0.02)
            chunks.append(hd); lens.append(hl)
            ids[n_rand:] = n_targets + np.arange(n_hom)
            n_targets += n_hom
        pairs.append(np.stack([np.full(targets_per_query, qi, np.int64), ids], 1))
    to = np.zeros(n_targets + 1, np.uint64)
    to[1:] = np.cumsum(np.concatenate(lens))
    return queries, np.concatenate(chunks), to, np.concatenate(pairs).astype(np.uint32)


class ClockSampler:
    """nvidia-smi SM clock + throttle reasons, sampled while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.thread = index, [], False, None

    def _run(self):
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.samples.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def start(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=6)
        sm, mx, reasons = [], 0.0, set()
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx = max(mx, float(s[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_int_peak():
    """thread-instructions/clk/SM of the DPX instructions, measured live on this GPU by the microbenchmark."""
    exe = os.path.join(ROOT, "profiles", "microbench", "int_pipe_rate")
    src = exe + ".cu"
    try:
        if not os.path.exists(exe):
            subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-o", exe, src])
        out = subprocess.run([exe], capture_output=True, text=True, timeout=120).stdout
        rates = {}
        for line in out.splitlines():
            parts = line.split()
            if len(parts) > 2 and "thread-instr/clk/SM" in line:
                rates[parts[0]] = float(line.split("thread-instr/clk/SM")[0].split()[-1])
        return rates, "measured live by profiles/microbench/int_pipe_rate"
    except Exception as e:  # pragma: no cover
        return {}, "microbenchmark unavailable: %r" % (e,)


def cpu_info():
    """what the host really offers: affinity mask, cgroup quota, model -- os.cpu_count() alone overstates a restricted box"""
    info = {"os_cpu_count": os.cpu_count(), "affinity_cpus": len(os.sched_getaffinity(0))}
    try:
        info["cpu_model"] = [l.split(":", 1)[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")][0]
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            info["cgroup_" + os.path.basename(path)] = open(path).read().strip()
        except Exception:
            pass
    threads = info["affinity_cpus"]
    try:   # cgroup v2 quota "max 100000" or "<quota> <period>"
        q, per = info.get("cgroup_cpu.max", "max 100000").split()
        if q != "max":
            threads = max(1, min(threads, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    info["threads_used"] = threads
    return info


class CpuScan:
    """The reference's ungapped_alignment on the host cores the way runFilterOnCpu runs it: one persistent thread team with one
    SmithWaterman per thread (oracle/_ref: ref_scan_init / ref_scan_batch), or the C port when oracle/_ref is absent."""

    def __init__(self, res, off, threads):
        from oracle.pyoracle import Oracle, Ref
        self.res, self.off64, self.threads = res, np.ascontiguousarray(off, np.int64), threads
        self.kind = "reference" if Ref.available() else "port"
        self.max_len = int((self.off64[1:] - self.off64[:-1]).max())
        if self.kind == "reference":
            self.ref = Ref()
            self.team = self.ref.scan_team(max(self.max_len, 1024), True, threads)
        else:
            mat, pb = load_matrix()
            self.orc = Oracle(mat, pb)

    def scan(self, queries, n_targets=None):
        """-> u8/int32 scores [nq][n]"""
        toff = self.off64 if n_targets is None else self.off64[:n_targets + 1]
        if self.kind == "reference":
            return self.ref.scan_batch(self.team, queries, self.res, toff)
        out = []
        for q in queries:
            cb, bias = self.orc.query_cb(q, True)
            out.append(self.orc.ungapped(q, cb, bias, self.res, toff, nthreads=self.threads, fast=True))
        return np.stack(out)

    def close(self):
        if self.kind == "reference":
            self.ref.scan_free(self.team)


def hit_list_from_scores(scores, thr, k):
    """the filter/sort/truncate of runFilterOnCpu (ungappedprefilter.cpp:450-478): score > thr, (score desc, id asc), first k"""
    ids = np.nonzero(scores > thr)[0]
    order = np.lexsort((ids, -scores[ids].astype(np.int64)))[:k]
    return ids[order].astype(np.uint32), scores[ids[order]].astype(np.int32)


def cpu_reference_gcups(batch_queries, res, off, budget_s, gpu_dense=None, gpu_hits=None, thr=15, max_hits=300):
    """cpu_baseline of the scan: the same query batches as the GPU arm, whole DB, all usable host threads, until the budget is spent;
    plus a 1-thread figure on a bounded sample, and the at-scale parity check: the reference's scores of every target (and the hit
    lists they imply) for the queries it got through, against what the GPU produced for the same queries."""
    ci = cpu_info()
    threads = ci["threads_used"]
    off64 = np.ascontiguousarray(off, np.int64)
    db_res = float(off64[-1])
    one = CpuScan(res, off, 1)
    n1 = int(min(len(off64) - 1, 40000))
    one.scan(batch_queries[0][:1], 2000)
    t0 = time.perf_counter()
    one.scan(batch_queries[0][:1], n1)
    gc1 = len(batch_queries[0][0]) * float(off64[n1]) / 1e9 / (time.perf_counter() - t0)
    one.close()
    cs = CpuScan(res, off, threads)
    cs.scan(batch_queries[0][:1], min(len(off64) - 1, 20000))      # warm: page in, spin up the team
    cells, dt, nq, same_scores, same_hits, checked = 0.0, 0.0, 0, True, True, 0
    for bi, qs in enumerate(batch_queries):
        pos = 0
        while pos < len(qs) and dt < budget_s:
            part = qs[pos:pos + 4]
            t0 = time.perf_counter()
            sc = cs.scan(part)
            dt += time.perf_counter() - t0
            cells += float(sum(len(q) for q in part)) * db_res
            if gpu_dense is not None and bi < len(gpu_dense):
                for k in range(len(part)):
                    same_scores &= bool(np.array_equal(sc[k].astype(np.uint8), gpu_dense[bi][pos + k]))
                    if gpu_hits is not None:
                        ids, scs = hit_list_from_scores(sc[k].astype(np.int32), thr, max_hits)
                        gi, gs = gpu_hits[bi][pos + k]
                        same_hits &= bool(np.array_equal(ids, gi) and np.array_equal(scs, gs))
                    checked += 1
            pos += len(part)
            nq += len(part)
        if dt >= budget_s:
            break
    cs.close()
    out = {"value": cells / 1e9 / dt, "unit": METRIC, "cores": threads, "kind": cs.kind, "gcups_1_thread": gc1, "host": ci,
           "sample": "%d queries (the GPU arm's own batches, in order) x whole %d-sequence DB = %.3g cells in %.1f s; 1-thread figure on "
                     "1 query x %d targets; persistent thread team, one SmithWaterman per thread" % (nq, len(off64) - 1, cells, dt, n1)}
    if gpu_dense is not None:
        out["scan_identical_to_gpu"] = bool(same_scores) and checked > 0
        out["hit_lists_identical_to_gpu"] = bool(same_hits) and checked > 0
        out["queries_compared_with_gpu"] = checked
        out["scores_compared_with_gpu"] = checked * (len(off64) - 1)
    return out


def cpu_reference_align_step(queries, tdata, toff, lists, gpu_results, gpu_pool, budget_s, threads):
    """The reference's Matcher::getSWResult loop + resultToBuffer (oracle/_ref: ref_align_query, one query per call, one call
    per host thread) on as many of the same prefilter lists as fit the time budget; also checks the records against the GPU's."""
    from concurrent.futures import ThreadPoolExecutor
    from mmseqs2_b200 import alignment as al
    from oracle.pyoracle import Ref
    if not Ref.available():
        return {"unavailable": "oracle/_ref not built"}
    ref = Ref()
    to64 = np.ascontiguousarray(toff, np.int64)
    db_res = int(to64[-1])

    def one(qi):
        return ref.align_query(queries[qi], qi, tdata, to64, lists[qi], lists[qi], db_res, sw_mode=2, eval_thr=1e-3)

    t0 = time.perf_counter()
    one(0)
    per_query = max(1e-4, time.perf_counter() - t0)
    n = int(min(len(queries), max(threads, budget_s * threads / per_query / 4)))
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        outs = list(ex.map(one, range(n)))
    dt = time.perf_counter() - t0
    n_aln = sum(o[1] for o in outs)
    same = all(al.records(gpu_results[qi], gpu_pool, True, True) == outs[qi][0] for qi in range(n))
    return {"value": n_aln / dt, "unit": "alignments/s", "cores": threads, "kind": "reference",
            "sample": "%d of the %d lists (%d alignments) in %.1f s" % (n, len(queries), n_aln, dt), "records_identical_to_gpu": bool(same)}


def cpu_reference_sw(queries, td, to, pairs, budget_s, threads):
    """alignScoreEndPos of the reference over a bounded prefix of the pair list, one OpenMP region over queries with one
    SmithWaterman object per thread (the shape of Alignment::run); falls back to the C port when oracle/_ref is absent"""
    from oracle.pyoracle import Oracle, Ref
    mat, pb = load_matrix()
    to64 = to.astype(np.int64)
    cells_pair = np.array([len(queries[a]) * int(to64[b + 1] - to64[b]) for a, b in pairs], np.float64)
    if Ref.available():
        ref = Ref()
        per_q = max(1, len(pairs) // len(queries))
        probe = pairs[pairs[:, 0] < min(len(queries), 2 * threads)]
        t0 = time.perf_counter()
        ref.sw_score_endpos_multi(queries, True, td, to64, probe, nthreads=threads)
        rate = cells_pair[:len(probe)].sum() / max(time.perf_counter() - t0, 1e-3)
        want_pairs = int(np.searchsorted(np.cumsum(cells_pair), rate * budget_s))
        nq = int(min(len(queries), max(2 * threads, want_pairs // per_q)))
        sub = pairs[pairs[:, 0] < nq]
        t0 = time.perf_counter()
        ref.sw_score_endpos_multi(queries, True, td, to64, sub, nthreads=threads)
        dt = time.perf_counter() - t0
        cells = float(cells_pair[:len(sub)].sum())
        kind = "reference"
    else:
        orc = Oracle(mat, pb)
        cells, dt, nq = 0.0, 0.0, 0
        for qi in range(len(queries)):
            if dt >= budget_s:
                break
            tl = pairs[pairs[:, 0] == qi][:, 1]
            sd, so = td[int(to64[tl[0]]):int(to64[tl[-1] + 1])], to64[tl[0]:tl[-1] + 2] - to64[tl[0]]
            cb, bias = orc.query_cb(queries[qi], True)
            t0 = time.perf_counter()
            orc.sw_score_endpos(queries[qi], cb, bias, sd, so, nthreads=threads)
            dt += time.perf_counter() - t0
            cells += float(len(queries[qi])) * float(so[-1])
            nq += 1
        kind = "port"
    return {"value": cells / 1e9 / dt, "unit": METRIC, "cores": threads, "kind": kind,
            "sample": "alignScoreEndPos, first %d queries x their target lists = %.3g cells in %.1f s" % (nq, cells, dt)}


def run_reference_arm(args):
    """--impl reference: the reference's own CPU scorer on the same workload and the same step shape as the GPU arm (one step = one
    batch of queries_per_step queries against the whole DB; the two batches alternate), all usable host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ci = cpu_info()
    threads = ci["threads_used"]
    n_distinct = 2
    res, off, queries = make_scan_workload(0, args.db_seqs, args.queries_per_step, n_distinct)
    batches = [queries[b * args.queries_per_step:(b + 1) * args.queries_per_step] for b in range(n_distinct)]
    db_res = float(np.asarray(off, np.int64)[-1])
    cs = CpuScan(res, off, threads)
    cs.scan(batches[0][:1], min(len(off) - 1, 20000))
    times, cells_done = [], 0.0
    for s in range(args.warmup + args.steps):
        qs = batches[s % n_distinct]
        t0 = time.perf_counter()
        cs.scan(qs)
        dt = time.perf_counter() - t0
        if s >= args.warmup:
            times.append(dt); cells_done += float(sum(len(q) for q in qs)) * db_res
    cs.close()
    total = sum(times)
    val = cells_done / 1e9 / total
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": METRIC, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / max(1, len(times)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": scan_config(args, int(db_res), 1),
            "cpu_baseline": {"value": val, "unit": METRIC, "cores": threads, "kind": cs.kind, "host": ci,
                             "sample": "%d steps x %d queries x whole DB (%.3g cells per step)" % (len(times), args.queries_per_step, cells_done / max(1, len(times)))},
            "e2e": {"value": val, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


def dump_scan_outputs(out_dir, hits, n_hits):
    """What a caller of the scan job receives: per query the hit count and the (target id, score) list.  Slots past a query's
    hit count are set to -1, so that equal results give equal files."""
    valid = np.arange(hits.shape[1])[None, :] < n_hits[:, None].astype(np.int64)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "scan_n_hits.npy"), n_hits.astype(np.float64))
    np.save(os.path.join(out_dir, "scan_hit_ids.npy"), np.where(valid, hits["id"], -1).astype(np.float64))
    np.save(os.path.join(out_dir, "scan_hit_scores.npy"), np.where(valid, hits["score"], -1).astype(np.float32))


def scan_config(args, db_residues, world):
    return {"workload": "ungapped prefilter (BASELINE config[1]): L~350 protein queries vs %d-seq synthetic DB "
                        "(log-normal lengths, %d residues), BLOSUM62 + composition bias; a step = %d queries x the whole DB "
                        "(a sample of the 10k-query job: the rate does not depend on the number of steps)" % (args.db_seqs, db_residues, args.queries_per_step),
            "queries_per_step_per_gpu": args.queries_per_step, "db_seqs": args.db_seqs, "max_hits": args.max_hits,
            "parallelism": "query-sharded x%d, DB replicated" % world,
            "l2": "target DB (%d MB) larger than L2; two alternating query batches" % (db_residues >> 20)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--db-seqs", type=int, default=1000000)
    ap.add_argument("--queries-per-step", type=int, default=16)
    ap.add_argument("--max-hits", type=int, default=300)
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--sw-queries", type=int, default=1024)     # x --sw-targets = 1 M pairs: BASELINE config[2]
    ap.add_argument("--sw-targets", type=int, default=1024)
    ap.add_argument("--no-libmarv", action="store_true", help="skip the reference's own GPU scorer (baseline/_ref) on the same DB")
    ap.add_argument("--search-wallclock", type=int, default=0, metavar="Q",
                    help="also run `mmseqs search` through the patched reference host vs the AVX2 build on Q queries (integration/search_wallclock.py)")
    ap.add_argument("--nucl-reads", type=int, default=200000)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=20.0, help="seconds of CPU work for the scan's cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the hit lists of the last timed step (rank 0's queries) to DIR/*.npy, to compare two builds")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.dump_outputs and (args.impl != "b200" or args.steps < 1):
        ap.error("--dump-outputs needs --impl b200 and at least one timed step")

    if args.impl == "reference":
        run_reference_arm(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    import torch
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from mmseqs2_b200 import Context, SubMatrix
    mat, pb = load_matrix()
    sm = SubMatrix(mat, pb)
    ctx = Context(local_rank)
    info = ctx.device_info()

    n_distinct = 2  # alternate between two query batches so no step re-reads the previous step's profiles
    res, off, queries = make_scan_workload(rank, args.db_seqs, args.queries_per_step, n_distinct)
    ctx.load_db(res, off, 21)
    db_residues = int(off[-1])
    batches, batch_seqs = [], []
    for b in range(n_distinct):
        qs = queries[b * args.queries_per_step:(b + 1) * args.queries_per_step]
        batches.append([sm.ssw_query(q) for q in qs])
        batch_seqs.append(qs)
    jobs = [ctx.scan_job(bt, 15, args.max_hits) for bt in batches]
    cells_per_step = [j.cells for j in jobs]

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- value: resident inputs, device-timed -------------------------------------------------------
    # N=1: scans back to back on the library's stream, CUDA events around the loop.
    # N>1: the same, plus per step the hit lists of every rank gathered with one NCCL all_gather -- pipelined: two scans stay in flight
    #      while the lists of the oldest finished step are downloaded (on the job's own event) and gathered on a second stream.
    pipe_jobs = jobs if dist is None else jobs + [ctx.scan_job(batches[0], 15, args.max_hits)]
    pipe_cells = cells_per_step if dist is None else cells_per_step + [cells_per_step[0]]
    gather = None
    if dist is not None:
        from mmseqs2_b200.sharding import HitGather
        gather = HitGather(args.queries_per_step, args.max_hits, dist, torch.device("cuda", local_rank))
    npj = len(pipe_jobs)

    def run_steps(n_steps):
        cells = 0
        if dist is None:
            for s in range(n_steps):
                pipe_jobs[s % npj].run()
                cells += pipe_cells[s % npj]
            return cells
        depth = 2
        for s in range(min(depth, n_steps)):
            pipe_jobs[s % npj].run()
        for s in range(n_steps):
            h, nh, _ = pipe_jobs[s % npj].fetch()          # waits for step s only
            if s + depth < n_steps:
                pipe_jobs[(s + depth) % npj].run()         # its buffers were read out one iteration ago
            if len(gather.started) >= 2:
                gather.finish()
            gather.start(h, nh)
            cells += pipe_cells[s % npj]
        gather.drain()
        return cells

    run_steps(args.warmup)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:          # the line is rank 0's; eight ranks forking nvidia-smi ten times a second only load the host
        sampler.start()
    launches0 = ctx.launches
    ctx.event_record(0)
    t_wall0 = time.perf_counter()
    total_cells = run_steps(args.steps)
    ctx.event_record(1)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    dev_ms = ctx.event_elapsed_ms(0, 1)
    launches = ctx.launches - launches0
    clocks = sampler.stop() if rank == 0 else {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    step_ms = (t_wall * 1e3 if dist is not None else dev_ms)
    if args.dump_outputs and rank == 0:
        dump_scan_outputs(args.dump_outputs, *pipe_jobs[(args.steps - 1) % npj].fetch()[:2])
    # kernel-only time of the scan kernel for the roofline (events around the launches of one job, no fetch)
    ctx.event_record(2)
    jobs[0].run()
    ctx.event_record(3)
    kern_ms = ctx.event_elapsed_ms(2, 3)

    # ---- e2e: host buffers through the public call ----------------------------------------------------
    # N>1: the hit lists of every step are gathered as in the `value` loop (same collective, started after the call returns and
    # finished a step later), so the first timed step does not pay NCCL's lazy set-up of another collective type.
    def e2e_step(s):
        h, nh, _ = ctx.ungapped_scan(batches[s % n_distinct], 15, args.max_hits)
        if gather is not None:
            if len(gather.started) >= 2:
                gather.finish()
            gather.start(h, nh)

    for s in range(min(2, args.warmup)):
        e2e_step(s)
    if gather is not None:
        gather.drain()
    barrier()
    t0 = time.perf_counter()
    e2e_cells = 0
    for s in range(args.steps):
        e2e_step(s)
        e2e_cells += cells_per_step[s % n_distinct]
    if gather is not None:
        gather.drain()
    barrier()
    e2e_s = time.perf_counter() - t0
    h2d = sum(p.profile.nbytes for p in batches[0])
    d2h = len(batches[0]) * (args.max_hits * 8 + 4)

    # what the GPU produced for both batches (every target's score + the hit lists), kept for the at-scale parity check of the
    # cpu_baseline leg; fetched now because the secondaries below load other DBs into the context
    gpu_dense, gpu_hits = [], []
    if rank == 0 and world == 1 and not args.no_cpu:
        for j in jobs:
            j.run()
            h, nh, dn = j.fetch(want_dense=True)
            gpu_dense.append(dn)
            gpu_hits.append([(h[i]["id"][:int(nh[i])].copy(), h[i]["score"][:int(nh[i])].copy()) for i in range(len(h))])

    # ---- reduce over ranks (max time, sum cells) ---------------------------------------------------------
    if dist is not None:
        t = torch.tensor([step_ms, e2e_s, float(total_cells), float(e2e_cells)], dtype=torch.float64, device="cuda")
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        step_ms, e2e_s = float(tmax[0]), float(tmax[1])
        total_cells, e2e_cells = float(tsum[2]), float(tsum[3])
    value = total_cells / 1e9 / (step_ms / 1e3)
    e2e_value = e2e_cells / 1e9 / e2e_s

    line = {"metric": METRIC, "value": value, "unit": METRIC, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "s16x2", "data": "synthetic",
            "config": scan_config(args, db_residues, world),
            "e2e": {"value": e2e_value, "unit": METRIC, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches), "clocks": clocks, "device": info}

    if rank == 0:
        # ---- roofline of the dominant kernel (ungapped_scan_kernel) ----------------------------------------
        rates, how = measured_int_peak()
        dpx = rates.get("viaddmin_s16x2_relu") or rates.get("viaddmax_s16x2_relu")
        clk_mhz = clocks.get("sm_mhz") or 1965.0
        cells_job0 = cells_per_step[0]
        achieved_ops = cells_job0 * SCAN_OPS_PER_CELL / (kern_ms / 1e3) / 1e12
        roof = {"bound": "int-pipe", "kernel": "ungapped_scan_kernel", "achieved": achieved_ops, "unit": "T thread-instr/s",
                "ops_per_cell": SCAN_OPS_PER_CELL, "kernel_ms": kern_ms, "kernel_gcups": cells_job0 / 1e9 / (kern_ms / 1e3),
                "peak": None, "frac": None, "traffic": None, "peak_source": how,
                "hbm": {"achieved_gbs": (len(batches[0]) * (db_residues + args.db_seqs)) / 1e9 / (kern_ms / 1e3),
                        "peak_gbs": None, "note": "algorithmic bytes = DB residues read once per query + 1 B score per target"}}
        try:
            pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            roof["hbm"]["peak_gbs"] = pk.get("hbm_gbs")
            roof["hbm"]["frac"] = roof["hbm"]["achieved_gbs"] / pk["hbm_gbs"]
        except Exception:
            roof["hbm"]["peak_gbs"] = 6650.0
            roof["hbm"]["peak_source"] = "fallback"
        try:   # DRAM traffic of the dominant launch, from the committed ncu capture of this same command
            tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))["dominant"]
            roof["traffic"] = tr["dram_bytes_read"] + tr["dram_bytes_write"]
            roof["traffic_note"] = "bytes of the longest scan launch of a step, %s (%d of the 16 queries), ncu capture in profiles/; algorithmic %d" % (
                tr["kernel"], tr["queries_in_launch"], tr["algorithmic_bytes"])
        except Exception:
            pass
        if dpx:
            peak = dpx * info["sm_count"] * clk_mhz * 1e6 / 1e12
            roof["peak"] = peak
            roof["frac"] = achieved_ops / peak
            roof["dpx_thread_instr_per_clk_per_sm"] = dpx
            roof["clock_mhz_used"] = clk_mhz
        # the resource that actually binds (DESIGN 3.1, ncu: l1tex data-pipe wavefronts 92-98 % of peak): 2 B of profile per cell through
        # the 128 B/clk/SM shared-memory pipe (LDS.128 measured at 8.0 per clk per SM by the same microbenchmark)
        lds = rates.get("LDS.128")
        smem_peak_gcups = (lds or 8.0) * 16.0 / 2.0 * info["sm_count"] * clk_mhz * 1e6 / 1e9
        roof["binding_resource"] = {"name": "shared-memory pipe", "bytes_per_cell": 2.0, "lds128_per_clk_per_sm": lds or 8.0,
                                    "peak_gcups": smem_peak_gcups, "frac": roof["kernel_gcups"] / smem_peak_gcups}
        line["roofline"] = roof

        # ---- secondary: the whole hot path of `search --prefilter-mode 1` for one query batch, host buffers end to end:
        #      ungapped scan of the DB -> top hits -> gapped score of every hit -> score gate -> end/start positions of survivors
        if not args.no_secondary and world == 1:
            try:
                from mmseqs2_b200 import alignment as al
                evp = al.EvalueParams.defaults("blosum62.out", 11, 1, db_residues)
                apar = al.AlignParams(sw_mode=al.SCORE_COV_SEQID, eval_thr=1e-3)      # what easy-search runs: -a, -e 1e-3

                def search_once(bt, qseqs):
                    h, nh, _ = ctx.ungapped_scan(bt, 15, args.max_hits)
                    lists = [h[qi]["id"][:int(nh[qi])] for qi in range(len(bt))]
                    res, pool, n_aln = al.align_batch(ctx, sm, qseqs, lists, apar, evp)
                    return n_aln, sum(len(r) for r in res), res

                search_once(batches[0], batch_seqs[0])
                search_once(batches[1], batch_seqs[1])     # both batches once: the device buffer pool has its steady-state sizes
                t0 = time.perf_counter()
                n_pairs, n_surv, _ = search_once(batches[1], batch_seqs[1])
                sdt = time.perf_counter() - t0
                line.setdefault("secondary", {})["search_pipeline"] = {
                    "workload": "prefilter + align for %d queries vs the %d-seq DB, host buffers, one batch: ungapped scan -> top-%d hit lists -> "
                                "b200_align_batch (-a, -e 1e-3: gapped score/end, E-value + coverage gate, start, CIGAR, criteria, order)"
                                % (len(batches[1]), args.db_seqs, args.max_hits),
                    "queries_per_s": len(batches[1]) / sdt, "ms": sdt * 1e3, "prefilter_hits": int(n_pairs), "accepted_alignments": int(n_surv),
                    "GCUPS_scan_equivalent": cells_per_step[1] / 1e9 / sdt}
            except Exception as e:  # pragma: no cover
                line.setdefault("secondary", {})["search_pipeline"] = {"error": repr(e)}

        # ---- secondary: gapped SW rescoring (config[2] shape) ------------------------------------------------
        if not args.no_secondary and world == 1:
            try:
                sq, std, sto, spairs = make_sw_workload(args.sw_queries, args.sw_targets)
                ctx.load_db(std, sto, 21)
                sprofs = [sm.ssw_query(q) for q in sq]
                resid = float(sum(len(sq[a]) + int(sto[b + 1] - sto[b]) for a, b in spairs))
                clk = ClockSampler(local_rank); clk.start()
                # (a) score-only fast path: sw16_kernel (two targets per warp, int16x2)
                fjob = ctx.sw_score_job(sprofs, spairs)
                fjob.run(); ctx.sync()
                ctx.event_record(4)
                for _ in range(3):
                    fjob.run()
                ctx.event_record(5)
                f_ms = ctx.event_elapsed_ms(4, 5) / 3
                ctx.sw_score(sprofs, spairs)          # first full-size call grows the device buffer pool
                t0 = time.perf_counter()
                sc_host = ctx.sw_score(sprofs, spairs)
                f_e2e = time.perf_counter() - t0
                sw_cells = fjob.cells
                sc_job = fjob.fetch()
                fjob.close()
                # (b) score + end positions: sw32_kernel (one pair per warp, int32)
                sjob = ctx.sw_job(sprofs, spairs)
                sjob.run(); ctx.sync()
                ctx.event_record(6)
                sjob.run()
                ctx.event_record(7)
                sw_ms = ctx.event_elapsed_ms(6, 7)
                ends = sjob.fetch()
                sjob.close()
                ctx.sw_score_endpos(sprofs, spairs)
                t0 = time.perf_counter()
                ends_host = ctx.sw_score_endpos(sprofs, spairs)   # packed score pass + packed FIND pass, host buffers
                se_e2e = time.perf_counter() - t0
                assert np.array_equal(ends_host, ends)
                ctx.sw_align(sprofs, spairs)
                t0 = time.perf_counter()
                aln_host = ctx.sw_align(sprofs, spairs)   # score -> end -> start positions, three chained packed launches
                al_e2e = time.perf_counter() - t0
                assert np.array_equal(aln_host["score"], ends["score"]) and np.array_equal(aln_host["dbend"], ends["dbend"])
                sclk = clk.stop()
                assert np.array_equal(sc_job, ends["score"]) and np.array_equal(sc_host, sc_job)
                sclk_mhz = sclk.get("sm_mhz") or clk_mhz
                sec = {"workload": "gapped SW rescoring (BASELINE config[2] shape): %d pairs, L log-uniform 50-2000, "
                                   "BLOSUM62 gap 11/1, half random / half homologs at 20-90%% identity" % len(spairs),
                       "value": sw_cells / 1e9 / (f_ms / 1e3), "unit": METRIC, "kernel": "sw16_kernel (score only)",
                       "ms": f_ms, "aligned_residues_per_s": resid / (f_ms / 1e3),
                       "e2e": {"value": sw_cells / 1e9 / f_e2e, "unit": METRIC,
                               "h2d_bytes": int(sum(p.profile.nbytes for p in sprofs) + spairs.nbytes), "d2h_bytes": int(4 * len(spairs))},
                       "score_endpos": {"value": sw_cells / 1e9 / (sw_ms / 1e3), "unit": METRIC, "kernel": "sw32_kernel<1>", "ms": sw_ms,
                                        "e2e": {"value": sw_cells / 1e9 / se_e2e, "unit": METRIC,
                                                "path": "b200_sw_score_endpos: sw16 score pass + sw16 FIND pass (end positions), host buffers"}},
                       "align": {"e2e": {"value": sw_cells / 1e9 / al_e2e, "unit": METRIC, "ms": al_e2e * 1e3,
                                         "path": "b200_sw_align on every pair: sw16 score -> FIND -> reverse pass chained on the device "
                                                 "(score, qEnd, dbEnd, qStart, dbStart), host buffers"}},
                       "word_mode_pairs": int(ends["word"].sum()), "clocks": sclk}
                dpx16 = rates.get("viaddmax_s16x2")
                if dpx16:
                    pk = dpx16 * info["sm_count"] * sclk_mhz * 1e6 / 1e12
                    ach = sw_cells * SW16_OPS_PER_CELL / (f_ms / 1e3) / 1e12
                    sec["roofline"] = {"bound": "int-pipe", "achieved": ach, "peak": pk, "unit": "T thread-instr/s",
                                       "frac": ach / pk, "ops_per_cell": SW16_OPS_PER_CELL, "clock_mhz_used": sclk_mhz}
                i32 = rates.get("viaddmax_s32")
                if i32:
                    pk = i32 * info["sm_count"] * sclk_mhz * 1e6 / 1e12
                    ach = sw_cells * SW32_OPS_PER_CELL / (sw_ms / 1e3) / 1e12
                    sec["score_endpos"]["roofline"] = {"bound": "int-pipe", "achieved": ach, "peak": pk, "frac": ach / pk,
                                                       "ops_per_cell": SW32_OPS_PER_CELL}
                if not args.no_cpu:
                    sec["cpu_baseline"] = cpu_reference_sw(sq, std, sto, spairs, 10.0, cpu_info()["threads_used"])
                # (c) the whole `align` step for these lists: b200_align_batch (score/end -> E-value + coverage gate -> start -> CIGAR ->
                #     result assembly, criteria, ordering) and the records of Matcher::resultToBuffer, host buffers end to end
                try:
                    from mmseqs2_b200 import alignment as al
                    order = np.argsort(spairs[:, 0], kind="stable")
                    bounds = np.searchsorted(spairs[order, 0], np.arange(len(sq) + 1))
                    lists = [spairs[order[bounds[i]:bounds[i + 1]], 1] for i in range(len(sq))]
                    evp = al.EvalueParams.defaults("blosum62.out", 11, 1, int(sto[-1]))
                    apar = al.AlignParams(sw_mode=al.SCORE_COV_SEQID, eval_thr=1e-3)
                    al.align_batch(ctx, sm, sq, lists, apar, evp)
                    t0 = time.perf_counter()
                    ares, apool, n_aln = al.align_batch(ctx, sm, sq, lists, apar, evp)
                    a_dt = time.perf_counter() - t0
                    step = {"workload": "`align` step (-a, -e 1e-3) over the same %d prefilter lists: alignments with E-value gate, start "
                                        "positions and CIGAR for the survivors, criteria, ordering" % len(sq),
                            "alignments_per_s": n_aln / a_dt, "ms": a_dt * 1e3, "alignments": n_aln,
                            "accepted": int(sum(len(r) for r in ares)), "unit": "alignments/s", "GCUPS_equivalent": sw_cells / 1e9 / a_dt}
                    if not args.no_cpu:
                        step["cpu_baseline"] = cpu_reference_align_step(sq, std, sto, lists, ares, apool, 8.0, cpu_info()["threads_used"])
                    sec["align_step"] = step
                except Exception as e:  # pragma: no cover
                    sec["align_step"] = {"error": repr(e)}
                line.setdefault("secondary", {})["sw_rescoring"] = sec
                sjob.close()
            except Exception as e:  # pragma: no cover
                line.setdefault("secondary", {})["sw_rescoring"] = {"error": repr(e)}

        # ---- secondary: the reference's own GPU scorer (libmarv, built in place by baseline/Makefile) on the same DB and queries ----
        if not args.no_secondary and not args.no_libmarv and world == 1:
            try:
                from baseline import marv
                if marv.available():
                    # our context goes first: both libraries want the whole GPU
                    mq = batch_seqs[0] + batch_seqs[1]
                    mp = [p.profile for p in batches[0] + batches[1]]
                    tb, _ = marv.time_tables(res, off, mq, mp, tables=("as_shipped", "sm90_dpx"), max_seqs=args.max_hits)
                    line.setdefault("secondary", {})["libmarv"] = {
                        "what": "Marv::scan of the reference (lib/libmarv compiled for sm_100, one call per query as ungappedprefilter.cpp:207 does) "
                                "on the same %d-sequence DB and the same %d queries; as_shipped = the kernel table libmarv selects on cc 10.0 "
                                "(its sm_89 half2 table), sm90_dpx = its H100 short2/DPX table installed through setCustomKernelConfig_Gapless" % (args.db_seqs, len(mq)),
                        "GCUPS": tb, "b200_e2e_GCUPS": e2e_value,
                        "b200_over_libmarv_best": e2e_value / max(v["gcups_wall"] for v in tb.values())}
                else:
                    line.setdefault("secondary", {})["libmarv"] = {"unavailable": "baseline/_ref/libmarv_harness.so not built (make -C baseline)"}
            except Exception as e:  # pragma: no cover
                line.setdefault("secondary", {})["libmarv"] = {"error": repr(e)}

        # ---- secondary: A1, the per-diagonal scorer of the k-mer prefilter, batched over queries (b200_diag_score_batch) -----------
        if not args.no_secondary and world == 1:
            try:
                rng = np.random.default_rng(6)
                ctx.load_db(res, off, 21)
                nqd, per_q = 64, 50000
                dqs = (queries * ((nqd + len(queries) - 1) // len(queries)))[:nqd]
                dprofs = [sm.diag_query(q, sm.comp_bias(q)) for q in dqs]
                lens = np.diff(np.asarray(off, np.int64))
                lists = []
                cells = 0
                for q in dqs:
                    ids = rng.integers(0, len(lens), per_q).astype(np.uint32)
                    dg = rng.integers(-(lens[ids] - 1), len(q), per_q)                # a diagonal that meets the rectangle
                    L = np.where(dg >= 0, np.minimum(lens[ids], len(q) - dg), np.minimum(lens[ids] + dg, len(q)))
                    cells += int(L.sum())
                    lists.append((ids, (dg & 0xffff).astype(np.uint16)))
                ctx.diag_score_batch(dprofs[:4], lists[:4])
                t0 = time.perf_counter()
                ctx.diag_score_batch(dprofs, lists)
                ddt = time.perf_counter() - t0
                dk_ms = ctx.last_kernel_ms
                t0 = time.perf_counter()
                for i in range(8):
                    ctx.diag_score(dprofs[i], lists[i][0], lists[i][1])
                one_dt = (time.perf_counter() - t0) / 8
                nh = nqd * per_q
                dbytes = cells + nh * (7 + 1)       # SURVEY 8(d): diagonal length + 7 B hit record in + 1 B out per hit
                line.setdefault("secondary", {})["diag_score"] = {
                    "workload": "per-diagonal scorer (A1): %d queries x %d (target, diagonal) hits on the %d-sequence DB, one batched call" % (nqd, per_q, args.db_seqs),
                    "hits_per_s": nh / (dk_ms / 1e3), "kernel_ms": dk_ms, "cells": cells,
                    "e2e": {"hits_per_s": nh / ddt, "ms": ddt * 1e3, "per_query_calls_hits_per_s": per_q / one_dt},
                    "roofline": {"bound": "hbm", "achieved": dbytes / 1e9 / (dk_ms / 1e3), "unit": "GB/s", "peak": roof["hbm"]["peak_gbs"],
                                 "frac": dbytes / 1e9 / (dk_ms / 1e3) / roof["hbm"]["peak_gbs"],
                                 "note": "random gathers of ~%d-residue diagonals: latency bound; sectors fetched exceed the algorithmic bytes" % (cells // nh)}}
            except Exception as e:  # pragma: no cover
                line.setdefault("secondary", {})["diag_score"] = {"error": repr(e)}

        # ---- secondary: nucleotide gapped aligner (config[4] shape in miniature: 150-bp reads vs genome pieces) ------------
        if not args.no_secondary and world == 1:
            try:
                from mmseqs2_b200 import synth
                rng = np.random.default_rng(4)
                ntargets = [synth.nucl_genome(rng, 30000) for _ in range(200)]
                reads, ntasks = synth.nucl_reads(rng, ntargets, args.nucl_reads, 150, subst=0.02, indel=0.002)
                ntd, nto = synth.pack(ntargets)
                ctx.load_db(ntd, nto, 5)
                ctx.nucl_align(reads[:2000], ntasks[:2000], decode=False)
                packed_reads = synth.pack(reads)
                t0 = time.perf_counter()
                nout, ncig, nbt = ctx.nucl_align(packed_reads, ntasks, decode=False)
                ndt = time.perf_counter() - t0
                nk_ms = ctx.last_kernel_ms
                nsec = {"workload": "nucleotide gapped aligner (BASELINE config[4] shape): %d reads x 150 bp (2 %% subst, 0.2 %% indel) vs "
                                    "%d x 30 kbp targets, nucleotide.out, gap 5/2, zdrop 40, band 64" % (len(reads), len(ntargets)),
                        "e2e": {"value": len(reads) / ndt, "unit": "alignments/s", "includes": "H2D reads + tasks, kernel, D2H results + CIGAR ops"},
                        "aligned_residues_per_s": float((nout["qend"] - nout["qstart"] + 1).sum()) / ndt,
                        "kernel": "nucl_align_kernel", "kernel_ms": nk_ms, "value": len(reads) / (nk_ms / 1e3), "unit": "alignments/s",
                        "mean_score": float(nout["score"].mean())}
                # SURVEY 8(d) for A7: HBM/latency bound; algorithmic bytes = 2 * (150 + band 64) residues + 32 B result per read
                nbytes = len(reads) * (2 * (150 + 64) + 32)
                nsec["roofline"] = {"bound": "hbm", "achieved": nbytes / 1e9 / (nk_ms / 1e3), "unit": "GB/s", "peak": roof["hbm"]["peak_gbs"],
                                    "frac": nbytes / 1e9 / (nk_ms / 1e3) / roof["hbm"]["peak_gbs"], "bytes_per_read": 2 * (150 + 64) + 32,
                                    "note": "tiny DPs (150 x <=214 cells in band 64): the kernel is occupancy/latency bound, not bandwidth bound"}
                if not args.no_cpu:
                    from oracle.pyoracle import Ref
                    if Ref.available():
                        ref = Ref()
                        m = min(len(reads), 200000)
                        t0 = time.perf_counter()
                        rout = ref.nucl_align_batch(reads[:m], ntd, nto.astype(np.int64), ntasks[:m], nthreads=cpu_info()["threads_used"])
                        rdt = time.perf_counter() - t0
                        same = bool(np.array_equal(rout[:, :5], np.stack([nout[f][:m] for f in ("score", "qstart", "qend", "dbstart", "dbend")], 1)))
                        nsec["cpu_baseline"] = {"value": m / rdt, "unit": "alignments/s", "cores": cpu_info()["threads_used"], "kind": "reference",
                                                "sample": "%d reads in %.2f s" % (m, rdt), "results_identical_to_gpu": same}
                line.setdefault("secondary", {})["nucl_align"] = nsec
            except Exception as e:  # pragma: no cover
                line.setdefault("secondary", {})["nucl_align"] = {"error": repr(e)}

        # ---- CPU baseline (bounded sample, rank 0, N=1 only) ---------------------------------------------------
        if not args.no_cpu and world == 1:
            try:
                line["cpu_baseline"] = cpu_reference_gcups(batch_seqs, res, off, args.cpu_budget, gpu_dense, gpu_hits, 15, args.max_hits)
            except Exception as e:  # pragma: no cover
                line["cpu_baseline"] = {"error": repr(e)}
        if args.search_wallclock > 0 and world == 1:
            try:
                outp = os.path.join(ROOT, "gpurun_out", "search_wallclock_bench.json")
                subprocess.run([sys.executable, os.path.join(ROOT, "integration", "search_wallclock.py"), "--db-seqs", str(args.db_seqs),
                                "--queries", str(args.search_wallclock), "--cpu-queries", str(max(16, args.search_wallclock // 8)), "--out", outp],
                               check=True, capture_output=True, timeout=3000)
                line["search_wallclock"] = json.load(open(outp))
            except Exception as e:  # pragma: no cover
                line["search_wallclock"] = {"error": repr(e)}
        print(json.dumps(line))
    for j in pipe_jobs:
        j.close()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
