#!/usr/bin/env python
"""bench.py — aligned query bp/s of the LexicMap query-side search path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4|c5] [--dump-outputs DIR]

--config c2 (default; BASELINE.json configs[1], the driver's run): 10,000 synthetic 1-kb queries vs a 1,000-genome synthetic index
    (50 families x 20 members x 1 Mbp, SURVEY.md §8d generators, seeds 20260924/20260925), index written by lmi-tools with the reference's
    default options (20,000 masks, seed-desert filling). One "step" = one pass of the whole hot path (sketch -> seed probe -> chain ->
    pseudo-align -> extend+WFA -> rows) over the batch. N>1 (torchrun, one rank per GPU): image replicated, every rank searches its own
    10k-query batch (weak scaling by query), no data-path collective; one NCCL all-reduce of the per-rank counters at the end.
--config c3 (configs[2], the north-star shape): 10,000 x 5-kb queries vs 100,000 genomes x 200 kbp, GENOME-SHARDED over the N ranks: rank r
    indexes and holds genomes [r*G/N, (r+1)*G/N), every rank searches the whole batch against its shard, per-query genome counts (`hits`)
    are summed with one NCCL all-reduce inside the timed region (what `lexicmap utils merge-search-results` does offline), e-values use the
    total bases of all shards. LMG_C3_GENOMES / LMG_C3_QUERIES scale it down for rehearsals (the JSON says so).
--config c4 (configs[3]): the reference's simulated ONT reads (tests/golden/demo_long_reads_subset.fasta.gz, 31 reads up to 63 kb) vs
    tests/data/demo.lmi (the demo genomes' windows of tests/golden/, seeded filler elsewhere) with the reference's demo flags — the WFA-heavy path.
--config c5 (configs[4]): seed-lookup microbenchmark on a synthetic seeds-only image, range-partitioned by mask over the ranks.
--dump-outputs DIR: after the timed steps, rank 0 writes what its last timed step returned as DIR/<name>.npy (float64): for c2-c4 every
    numeric column of the HSP rows (hsp_<column>.npy; all rows up to 64 MB, else the rows of a seeded sample of whole queries) and the
    rows per query; for c5 the lookup counters. The inputs are seeded, so two builds can be compared file by file.

`value`   = sum of query bases / CUDA-event time of lmg_search_staged (queries already in HBM), max over ranks.
`e2e`     = same metric through lmg_search_batch with HOST buffers (H2D of the queries and D2H of all rows inside the timed region).
`roofline`= seed-lookup kernel (k_probe_find2): SURVEY.md §8d byte model / its CUDA-event time / measured HBM peak.
`cpu_baseline` = the C++ oracle port of the reference path (the Go reference cannot run here: no Go toolchain) on the host cores.
--impl reference times that same CPU port with all usable host threads on the same workload.
"""
import argparse
import json
import os


def usable_cpus():
    """threads this process may really use: the affinity mask, capped by the cgroup CPU quota (a 1-GPU lease of a big box exposes all
    cores in os.cpu_count() but schedules only a share of them: round 1's CPU arm oversubscribed 128 threads on such a box)"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    if quota:
        n = max(1, min(n, int(quota + 0.5)))
    return n, (os.cpu_count() or 1), quota


# torchrun exports OMP_NUM_THREADS=1; the host side of the library (and the index builder) use threads for list handling, so give every
# rank its share of the usable cores before any OpenMP runtime is loaded
_world = int(os.environ.get("WORLD_SIZE", 1))
_ncpu = usable_cpus()[0]
if os.environ.get("OMP_NUM_THREADS", "1") == "1":
    os.environ["OMP_NUM_THREADS"] = str(max(1, _ncpu // max(1, _world)))
os.environ.setdefault("NCCL_DEBUG", "WARN")
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORK = os.environ.get("LMG_BENCH_DIR", "/tmp/lmg_bench")
C2 = dict(families=int(os.environ.get("LMG_BENCH_FAMILIES", 50)), members=int(os.environ.get("LMG_BENCH_MEMBERS", 20)), genome_len=int(os.environ.get("LMG_BENCH_GLEN", 1000000)),
          n_queries=int(os.environ.get("LMG_BENCH_NQ", 10000)), query_len=int(os.environ.get("LMG_BENCH_QLEN", 1000)), genome_seed=20260924, query_seed=20260925)
C3 = dict(genomes=int(os.environ.get("LMG_C3_GENOMES", 100000)), members=100, genome_len=200000, n_queries=int(os.environ.get("LMG_C3_QUERIES", 10000)), query_len=5000, genome_seed=20260924, query_seed=20260925)
C5 = dict(masks=20000, per_mask=int(os.environ.get("LMG_C5_PER_MASK", 500000)), n_queries=int(os.environ.get("LMG_C5_QUERIES", 10000000)), seed=20260926)
LANES = int(os.environ.get("LMG_LANES", 0))   # 0 = the library's automatic choice (up to 6 for large batches)


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def tools():
    from lexicmap_b200 import build
    return build.build_tools()


def build_index(out, args):
    """lmi-tools index into `out` (atomic rename; replaces a partial directory left by an interrupted build)"""
    if os.path.exists(os.path.join(out, "info.toml")):
        return
    t = time.time()
    tmp = out + ".tmp%d" % os.getpid()
    subprocess.check_call([tools(), "index", "--out", tmp] + args)
    if os.path.isdir(out):
        import shutil
        shutil.rmtree(out)
    os.rename(tmp, out)
    log("index built in %.1fs -> %s" % (time.time() - t, out))


def synth_queries(index, path, n, length, seed):
    if not os.path.exists(path):
        subprocess.check_call([tools(), "synth-queries", "--index", index, "--n", str(n), "--len", str(length), "--seed", str(seed), "--out", path + ".tmp"])
        os.rename(path + ".tmp", path)
    return path


def ensure_c2(rank):
    name = "c2d_%dx%dx%d" % (C2["families"], C2["members"], C2["genome_len"])   # "d": desert-filled (the writer's and the reference's default)
    idx = os.path.join(WORK, name + ".lmi")
    os.makedirs(WORK, exist_ok=True)
    build_index(idx, ["--synth", "%d,%d,%d,%d,20" % (C2["families"], C2["members"], C2["genome_len"], C2["genome_seed"])])
    qf = synth_queries(idx, os.path.join(WORK, "%s_q%d_%d_r%d.fa" % (name, C2["n_queries"], C2["query_len"], rank)), C2["n_queries"], C2["query_len"], C2["query_seed"] + rank)
    return idx, qf


def c3_queries(world, part=None):
    """the C3 batch: `world` parts of n/world queries, part p cut from the genomes of shard p (so every shard owns the hits of its share of the
    batch); the parts are regenerated straight from the synthetic collection, no index needed. Returns the list of part files (all parts, or [part])."""
    fam = C3["genomes"] // C3["members"]
    files = []
    for p in (range(world) if part is None else [part]):
        f0, f1 = fam * p // world, fam * (p + 1) // world
        n = C3["n_queries"] * (p + 1) // world - C3["n_queries"] * p // world
        path = os.path.join(WORK, "c3d_q%d_%d_w%d_p%d.fa" % (C3["n_queries"], C3["query_len"], world, p))
        if not os.path.exists(path):
            subprocess.check_call([tools(), "synth-queries", "--synth", "%d,%d,%d,%d,20" % (fam, C3["members"], C3["genome_len"], C3["genome_seed"]), "--genome-range", "%d,%d" % (f0 * C3["members"], f1 * C3["members"]),
                                   "--n", str(n), "--len", str(C3["query_len"]), "--seed", str(C3["query_seed"] + p), "--out", path + ".tmp%d" % os.getpid()])
            os.rename(path + ".tmp%d" % os.getpid(), path)
        files.append(path)
    return files


def ensure_c3(rank, world):
    """shard `rank` of the 100,000-genome collection: families [f0, f1) of 1,000 families x 100 members; one .lmi per shard"""
    fam = C3["genomes"] // C3["members"]
    f0, f1 = fam * rank // world, fam * (rank + 1) // world
    name = "c3d_%dx%dx%d_s%dof%d" % (fam, C3["members"], C3["genome_len"], rank, world)
    idx = os.path.join(WORK, name + ".lmi")
    os.makedirs(WORK, exist_ok=True)
    build_index(idx, ["--synth", "%d,%d,%d,%d,20" % (fam, C3["members"], C3["genome_len"], C3["genome_seed"]), "--synth-range", "%d,%d" % (f0 * C3["members"], f1 * C3["members"]),
                      "--threads", os.environ["OMP_NUM_THREADS"]])
    return idx


class ClockSampler:
    """One long-lived `nvidia-smi -lms 200` (the profiling recipe's clocks line) running during the timed region; parsed afterwards.
    A single process instead of one spawn per sample keeps the driver's management lock out of the way of the timed CUDA calls."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu):
        self.gpu, self.proc, self.sm, self.max_sm, self.reasons = gpu, None, [], 0, set()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def finish(self):
        if self.proc is None:
            return
        try:
            self.proc.terminate()
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            try:
                self.proc.kill()
            except Exception:
                pass
            out = ""
        for line in out.splitlines():
            o = [x.strip() for x in line.split(",")]
            try:
                self.sm.append(float(o[0]))
                self.max_sm = float(o[1])
            except Exception:
                continue
            for n, v in zip(self.NAMES, o[2:]):
                if "Active" in v and "Not" not in v:
                    self.reasons.add(n)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm or None, "reasons": sorted(self.reasons)}


def probe_model_bytes(survivors, sum_log2, sum_hit_sectors, sum_values):
    """SURVEY.md §8(d), K2 per probe: 12 B (query k-mer + mask id) + 32 B (anchor-table sector) + 32 B x ceil(log2(n_a + 1)) binary-search
    sectors (n_a = entries of the probe's anchor run) + 32 B x ceil(16 h / 32) sectors of the h matched entries + 16 B per anchor written
    (matched values). Sector-granular because the access is random; independent of this implementation's layout."""
    return 12 * survivors + 32 * survivors + 32 * sum_log2 + 32 * sum_hit_sectors + 16 * sum_values


def probe_r01_bytes(cnt):
    """round 1's model (kept for continuity with BENCH_r01 / VERDICT): 24-B record + 32-B anchor sector per probe, 32 B per search step
    actually taken, 16 B per entry scanned, 48 B per hit record written"""
    return int(cnt[1]) * (24 + 32) + int(cnt[2]) * 32 + int(cnt[3]) * 16 + int(cnt[4]) * 48


def hbm_peak():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


def cpu_port_throughput(idx_dir, seqs, threads, target_s=12.0, params=None, whole=False):
    """C++ port of the reference path on `threads` host threads: a calibration pass over a few queries, then a sample sized for ~target_s
    (all queries when `whole` or when they fit the time)"""
    from oracle_binding import Oracle
    o = Oracle(idx_dir)
    kw = params or {}
    n0 = min(len(seqs), max(threads, 64))
    t = time.time()
    o.search(seqs[:n0], o.default_params(**kw), threads=threads)
    dt = max(time.time() - t, 1e-3)
    n = len(seqs) if whole else int(min(len(seqs), max(n0, n0 * target_s / dt)))
    t = time.time()
    rows, _, _ = o.search(seqs[:n], o.default_params(**kw), threads=threads)
    dt = time.time() - t
    bp = sum(len(s) for s in seqs[:n])
    o.close()
    return bp / dt, n, dt, len(rows)


DUMP_BYTES = 64 << 20


def dump_arrays(d, arrays):
    os.makedirs(d, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.asarray(v, dtype=np.float64))


def dump_rows(d, rows, nq):
    """every numeric HSP column as float64 plus the rows per query; above DUMP_BYTES only the rows of whole queries, taken in a seeded order
    while they fit, so that two builds with the same rows dump the same sample"""
    names = [f for f in rows.dtype.names if f not in ("pad", "pad0", "cigar_off")]
    per_q = np.bincount(rows["query"].astype(np.int64), minlength=nq)
    budget = DUMP_BYTES - 8 * nq
    if len(rows) * 8 * len(names) > budget:
        order = np.random.default_rng(20260927).permutation(nq)
        fits = order[np.cumsum(per_q[order]) * 8 * len(names) <= budget]
        rows = rows[np.isin(rows["query"], fits)]
    dump_arrays(d, dict({"rows_per_query": per_q}, **{"hsp_" + f: rows[f] for f in names}))
    log("dumped %d rows (%d columns) to %s" % (len(rows), len(names), d))


def cpu_desc(threads):
    n, total, quota = usable_cpus()
    return {"cores": threads, "cores_visible": total, "cores_usable": n, "cgroup_quota": quota}


def base_config(a, workload, extra):
    cfg = {"workload": workload, "lanes": LANES if LANES else "auto (up to 6 concurrent sub-batches per call)",
           "l2": "index image (>1 GB) and per-batch buffers exceed the 126 MB L2; no explicit flush", "index": "written by lmi-tools with the reference's default options: 20,000 masks, seed-desert filling (-D 100 -d 50)"}
    cfg.update(extra)
    return cfg


# ------------------------------------------------------------------------------------------------ search configs (c2, c3, c4)
def run_search(a, rank, world, local):
    import torch
    import lexicmap_b200
    from lexicmap_b200.api import pack_queries
    from oracle_binding import read_fasta
    cfgname = a.config
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    search_kw, total_bases_all = {}, None
    # the device's random 32-byte-sector read rate (the physical ceiling of a lookup made of dependent random sectors), measured before the image and the arenas fill the memory
    from lexicmap_b200.api import gather_bench
    gb = gather_bench(device=local, gbytes=8.0) if rank == 0 else None
    if cfgname == "c2":
        if rank == 0:
            ensure_c2(0)
        if dist:
            dist.barrier()
        idx_dir, qf = ensure_c2(rank)
        ids, seqs = read_fasta(qf)
        workload = "%d synthetic %d-bp queries vs %d-genome synthetic index (%dx%dx%d bp), %s" % (
            C2["n_queries"], C2["query_len"], C2["families"] * C2["members"], C2["families"], C2["members"], C2["genome_len"],
            "BASELINE.json configs[1]" if (C2["families"], C2["members"], C2["genome_len"], C2["n_queries"], C2["query_len"]) == (50, 20, 1000000, 10000, 1000) else "LMG_BENCH_* override (not a BASELINE.json config as is)")
        config = base_config(a, workload, {"queries_per_gpu": C2["n_queries"], "query_len": C2["query_len"], "genomes": C2["families"] * C2["members"], "masks": 20000,
                                           "sharding": "by query, index replicated" if a.gpus > 1 else "single GPU", "seeds": [C2["genome_seed"], C2["query_seed"]]})
        scaling = "weak"
    elif cfgname == "c3":
        # the shard indexes are written in LMG_C3_WAVES groups of ranks so that the scratch disk holds world / waves of them at a time
        # (a shard of 12,500 genomes is ~10 GB on disk; ranks other than 0 delete theirs once the image is in HBM)
        waves = max(1, int(os.environ.get("LMG_C3_WAVES", 1)))
        sim = int(os.environ.get("LMG_C3_SIM_WORLD", 0))   # profiling aid: one GPU does exactly the work of rank 0 of a `sim`-GPU run (shard 0 of `sim`, the whole batch)
        if sim > 1 and world == 1:
            world = sim
        idx_dir, idx = None, None
        for wv in range(waves):
            if rank % waves == wv:
                idx_dir = ensure_c3(rank, world)
                t0 = time.time()
                idx = lexicmap_b200.Index(idx_dir, device=local)
                log("rank %d: image resident in %.1fs (%.2f GB, %d keys, %d values) %s" % (rank, time.time() - t0, idx.info.image_bytes / 1e9, idx.info.seed_keys, idx.info.seed_values, idx.load_times()))
                if rank != 0 and waves > 1:
                    import shutil
                    shutil.rmtree(idx_dir, ignore_errors=True)
            if dist:
                dist.barrier()
        c3_queries(world, part=rank)   # every rank writes the part cut from its own shard's genomes, then all read all parts (same box)
        if dist:
            dist.barrier()
        ids, seqs = [], []
        for qf in c3_queries(world):
            i2, s2 = read_fasta(qf)
            ids += i2
            seqs += s2
        full = (C3["genomes"], C3["n_queries"]) == (100000, 10000)
        workload = "%d synthetic %d-bp queries vs %d-genome synthetic collection (%d bp each) genome-sharded over %d GPU(s), %s" % (
            C3["n_queries"], C3["query_len"], C3["genomes"], C3["genome_len"], world, "BASELINE.json configs[2] (10k-query headline)" if full else "REDUCED rehearsal of BASELINE.json configs[2]")
        config = base_config(a, workload, {"queries": C3["n_queries"], "query_len": C3["query_len"], "genomes": C3["genomes"], "genomes_per_gpu": C3["genomes"] // world, "masks": 20000,
                                           "sharding": "by genome: one index shard per GPU, every GPU searches the whole batch, NCCL all-reduce(sum) of the per-query genome counts", "seeds": [C3["genome_seed"], C3["query_seed"]]})
        scaling = "strong"
    else:   # c4
        from conftest import DEMO_INDEX, GOLD
        idx_dir = DEMO_INDEX
        if not os.path.exists(os.path.join(idx_dir, "info.toml")):
            raise SystemExit("tests/data/demo.lmi is missing: run __graft_entry__.build() in the build container")
        qf = os.path.join(GOLD, "demo_long_reads_subset.fasta.gz")
        ids, seqs = read_fasta(qf)
        rep = int(os.environ.get("LMG_C4_REPEAT", 8))   # the sample is repeated so that a step holds enough work to time
        seqs = seqs * rep
        search_kw = dict(min_qcov_hsp=70.0, top_n_genomes=5, top_n_chains=1)
        workload = "%d simulated ONT reads (%s x%d) vs the reference's 15 demo genomes (stored windows, seeded filler), flags of demo/README.md:365-368; BASELINE.json configs[3] on the demo index" % (len(seqs), os.path.basename(qf), rep)
        config = base_config(a, workload, {"queries_per_gpu": len(seqs), "genomes": 15, "masks": 20000, "sharding": "by query, index replicated" if a.gpus > 1 else "single GPU", "flags": search_kw})
        scaling = "weak"
    if cfgname != "c3":
        t0 = time.time()
        idx = lexicmap_b200.Index(idx_dir, device=local)
        log("rank %d: image resident in %.1fs (%.2f GB, %d keys, %d values) %s" % (rank, time.time() - t0, idx.info.image_bytes / 1e9, idx.info.seed_keys, idx.info.seed_values, idx.load_times()))
    if cfgname == "c3":   # e-values over the whole collection
        tb = torch.tensor([float(idx.info.input_bases)], device="cuda", dtype=torch.float64)
        if dist:
            dist.all_reduce(tb)
        total_bases_all = int(tb.item())
        idx.set_total_bases(total_bases_all)
    packed = pack_queries(seqs)
    total_bp = int(packed[1][-1])
    prm = idx.default_params(lanes=LANES, **search_kw)
    staged = idx.stage(packed=packed)
    nq = len(seqs)

    def sync_all():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    def hits_allreduce(rows):
        """genome-sharded search: per-query genome counts of this shard -> NCCL sum over the shards (merge-search-results.go:143-153)"""
        from lexicmap_b200.dist import shard_hit_counts, allreduce_hits
        return allreduce_hits(shard_hit_counts(rows, nq), device=torch.device("cuda", local))

    collect = cfgname == "c3"
    # ---- value leg: staged inputs
    for _ in range(a.warmup):
        r = idx.search_staged(staged, prm, collect="rows" if collect else False)
        if collect:
            hits_allreduce(r[0])
    sync_all()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = int(idx.timing()[1][15])
    ms_steps, stage_ms, probe_ms, nrows, wall_ms, e2e_lib_ms, e2e_stage, kern_ms, kcnt = [], np.zeros(8), [], 0, [], [], np.zeros(8), np.zeros(16), None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(a.steps):
        t = time.perf_counter()
        keep = collect or (a.dump_outputs and i == a.steps - 1)   # the rows are copied to the host after the library's timed region
        r = idx.search_staged(staged, prm, collect="rows" if keep else False)
        ms, cnt = idx.timing()
        extra = 0.0
        rows = r[0] if keep else None
        nrows = len(rows) if keep else r
        if collect:
            ev0.record()
            hits_allreduce(rows)
            ev1.record()
            torch.cuda.synchronize()
            extra = ev0.elapsed_time(ev1)
        ms_steps.append(ms[7] + extra)
        stage_ms += ms[:8]
        probe_ms.append(ms[8])
        wall_ms.append((time.perf_counter() - t) * 1e3)
        kern_ms += ms
        kcnt = cnt
    sync_all()
    if a.dump_outputs and rank == 0:
        dump_rows(a.dump_outputs, rows, nq)
    launches = (int(idx.timing()[1][15]) - launches0) // max(a.steps, 1)
    # ---- e2e leg: host buffers in, rows out, every step
    e2e_ms = []
    for i in range(a.warmup + a.steps):
        t = time.perf_counter()
        if collect:
            r = idx.search(None, prm, packed=packed, rows_only=True)
            hits_allreduce(r[0])
            nr = len(r[0])
        else:
            nr = idx.search_count(packed, prm)
        torch.cuda.synchronize()
        if i >= a.warmup:
            e2e_ms.append((time.perf_counter() - t) * 1e3)
            e2e_lib_ms.append(idx.timing()[0][9])
            e2e_stage += idx.timing()[0][:8]
    sampler.finish()
    t_val = float(np.mean(ms_steps))
    t_e2e = float(np.mean(e2e_ms))
    own_bp = float(total_bp) if scaling == "weak" else float(total_bp) / world   # strong scaling: every rank searched the same batch; count it once
    hits = torch.tensor([float(nrows), own_bp, t_val, t_e2e], device="cuda", dtype=torch.float64)
    if dist:  # the collective of the report: reduce the per-rank counters (NCCL over NVLink)
        tmax = hits[2:].clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(hits[:2], op=dist.ReduceOp.SUM)
        hits[2:] = tmax
    rows_all, bp_all, t_val, t_e2e = (float(x) for x in hits.tolist())
    if rank != 0:
        idx.free_staged(staged)
        if dist:
            dist.barrier()   # rank 0 still runs its statistics / CPU legs; leave together
            dist.destroy_process_group()
        return None
    # ---- roofline of the seed-lookup kernel: statistics pass (untimed) on a slice of the same batch
    ns = min(len(seqs), 2000)
    idx.anchors(seqs[:ns], idx.default_params(**{k: v for k, v in search_kw.items() if k in ("min_prefix",)}))
    _, cnt = idx.timing()
    scale = float(total_bp) / max(1, sum(len(s) for s in seqs[:ns]))
    sums = idx.probe_model()
    alg_bytes = probe_model_bytes(int(cnt[1]), sums[0], sums[1], sums[2]) * scale
    r01_bytes = probe_r01_bytes(cnt) * scale
    peak, peak_src = hbm_peak()
    t_probe = float(np.mean(probe_ms)) * 1e-3
    achieved = alg_bytes / t_probe / 1e9 if t_probe > 0 else 0.0
    traffic, traffic_src = None, None   # DRAM bytes of the kernel per step from the committed `ncu --set full` capture of this workload (profiles/), if present
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        if tr.get("config") == cfgname and tr.get("workload_queries") == nq:
            traffic = float(tr["dram_bytes_per_step"])   # per step, like algorithmic_bytes_per_step (a step launches the kernel once per lane)
            traffic_src = tr.get("capture")
    except Exception:
        pass
    # the same kernel alone on the GPU (one lane, so no other lane's kernels share the SMs / HBM during its launches)
    p1 = idx.default_params(lanes=1, **search_kw)
    iso, iso_rg = [], []
    for _ in range(3):
        idx.search_count(packed, p1)
        tm = idx.timing()
        iso.append(tm[0][8])
        iso_rg.append(tm[1][12] * 1e-3)
    t_iso = float(np.mean(iso[1:])) * 1e-3
    rg_iso_ms = float(np.mean(iso_rg[1:]))
    rg_ms = float(kcnt[12]) * 1e-3   # regrouping pass (probes bucketed by mask before the lookup kernel) of the last timed step, summed over the lanes
    # ---- CPU baseline on this box (bounded sample)
    threads = usable_cpus()[0]
    cpu_s = float(os.environ.get("LMG_BENCH_CPU_S", 15.0))   # 0 skips the CPU leg (parameter sweeps only; the default run always reports it)
    cpu_seqs = seqs
    if cfgname == "c3" and world > 1:   # the batch is part 0 | part 1 | ...: the CPU sample takes the parts in turn so that 1/world of it hits shard 0's genomes, as in the whole job
        per = len(seqs) // world
        cpu_seqs = [seqs[p * per + i] for i in range(per) for p in range(world)]
    cpu_bps, cpu_n, cpu_dt, _ = cpu_port_throughput(idx_dir, cpu_seqs, threads, target_s=cpu_s, params=search_kw) if cpu_s > 0 else (0.0, 0, 0.0, None)
    cpu_note = "%d of the %d queries, %.1fs (C++ port of the reference path; Go toolchain absent)" % (cpu_n, len(seqs), cpu_dt)
    if cfgname == "c3" and world > 1:
        cpu_bps /= world
        cpu_note += "; measured against shard 0 (1/%d of the genomes) and divided by %d: the whole job searches every query against every shard" % (world, world)
    config_lanes = int(kern_ms[12] / max(a.steps, 1) + 0.5)
    # second roofline record: the dominant kernel (WFA forward pass). Cells = wavefront cells computed; bytes = what it writes to HBM per cell.
    wfa_ms = float(kern_ms[11]) / max(a.steps, 1)
    out = {"metric": "aligned query bp/s", "value": bp_all / (t_val * 1e-3), "unit": "bp/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": t_val,
           "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "int64", "data": "synthetic" if cfgname != "c4" else "reference demo reads (simulated ONT)", "config": config,
           "e2e": {"value": bp_all / (t_e2e * 1e-3), "unit": "bp/s", "h2d_bytes_per_step": int(packed[0].nbytes + packed[1].nbytes), "d2h_bytes_per_step": int(nrows * 136), "ms_per_step": t_e2e},
           "gpu_launches": launches, "rows_per_step": rows_all,
           "stage_ms": {k: float(v) / a.steps for k, v in zip(["h2d", "sketch", "seed_probe", "chain", "pseudo_align", "extend_wfa", "host_finish", "total"], stage_ms)},
           "roofline": {"bound": "hbm", "kernel": "k_probe_find2 (seed index lookup of the surviving probes)", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_capture": traffic_src,
                        "model": "SURVEY.md §8d: per probe 12 + 32 + 32*ceil(log2(n_a+1)) + 32*ceil(16h/32) + 16*h_out bytes", "algorithmic_bytes_per_step": alg_bytes, "probes_per_step": float(cnt[1]) * scale, "kernel_ms_per_step": t_probe * 1e3, "launches_per_step": config_lanes,
                        "regroup": {"note": "the probes are bucketed by mask (histogram + scan + scatter kernels) right before the lookup kernel so that a warp searches one bucket; that pass is not part of the kernel time above",
                                    "ms_per_step": rg_ms, "ms_alone": rg_iso_ms, "frac_with_regroup": (alg_bytes / (t_probe + rg_ms * 1e-3) / 1e9 / peak) if t_probe > 0 else 0.0,
                                    "frac_alone_with_regroup": (alg_bytes / (t_iso + rg_iso_ms * 1e-3) / 1e9 / peak) if t_iso > 0 else 0.0},
                        "alone": {"kernel_ms": t_iso * 1e3, "achieved": alg_bytes / t_iso / 1e9 if t_iso > 0 else 0.0, "frac": (alg_bytes / t_iso / 1e9 / peak) if t_iso > 0 else 0.0, "note": "same batch through one lane: no concurrent kernels"},
                        "r01_model": {"note": "round 1's byte model (24+32 B per probe, 32 B per search step taken, 16 B per entry scanned, 48 B per hit): kept for continuity with BENCH_r01", "algorithmic_bytes_per_step": r01_bytes, "frac": (r01_bytes / t_probe / 1e9 / peak) if t_probe > 0 else 0.0},
                        "random_sector_ceiling": {"note": "measured rate of independent random 32-byte-sector reads over an 8-GB buffer (k_gather_bench): the rate a lookup with scattered probes is held to; with the probes regrouped by bucket most sectors hit in L2 and the kernel is not bound by it",
                                                  "gbs_at_32B": gb["gbs_at_32B"], "frac_of_streaming_peak": gb["gbs_at_32B"] / peak, "kernel_alone_vs_ceiling": (alg_bytes / t_iso / 1e9 / gb["gbs_at_32B"]) if t_iso > 0 else 0.0, "kernel_in_region_vs_ceiling": achieved / gb["gbs_at_32B"]},
                        "peak_source": peak_src},
           "roofline_wfa": {"bound": "issue", "kernel": "k_wfa_reg<4>/<8> + k_wfa_bt2, then k_wfa_fast + k_wfa_bt for what is left (wavefront alignment: forward pass and backtrace)", "kernel_ms_per_step": wfa_ms, "alignments_per_step": int(kcnt[9]), "share_of_kernel_time": None,
                            "note": "instruction-issue bound (ncu: issue-active ~78 %, DRAM < 15 % of peak); see profiles/ for the ncu capture"},
           "cpu_baseline": dict({"value": cpu_bps, "unit": "bp/s", "kind": "port", "sample": cpu_note}, **cpu_desc(threads)),
           "debug": {"lanes_used": config_lanes, "staged_call_wall_ms": float(np.mean(wall_ms)), "e2e_call_wall_ms_in_lib": float(np.mean(e2e_lib_ms)), "e2e_stage_ms": [float(x) / a.steps for x in e2e_stage],
                     "kernel_ms": {k: float(kern_ms[i]) / a.steps for k, i in [("wfa_prep+general", 10), ("wfa_fwd+bt", 11), ("extend", 13), ("pa_anchors", 14), ("pa_chain", 15)]},
                     "wfa_jobs": int(kcnt[9]), "wfa_fallback_first": int(kcnt[10]), "wfa_general_jobs": int(kcnt[11]), "probe_find_us": int(kcnt[13]), "probe_survivors": int(kcnt[1]), "probe_issued": int(kcnt[0]), "wfa_per_round": int(kcnt[14]),
                     "index_load_ms": idx.load_times(), "image_bytes": int(idx.info.image_bytes), "total_bases_all_shards": total_bases_all},
           "clocks": sampler.summary()}
    idx.free_staged(staged)
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return out


# ------------------------------------------------------------------------------------------------ c5: seed-lookup microbenchmark
def run_c5(a, rank, world, local):
    import torch
    import lexicmap_b200
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    m, per, nq = C5["masks"], C5["per_mask"], C5["n_queries"]
    from lexicmap_b200.api import gather_bench
    gb = gather_bench(device=local, gbytes=8.0) if rank == 0 else None   # the device's random 32-byte-sector read rate, measured before the index fills the memory
    lo, hi = m * rank // world, m * (rank + 1) // world
    free_b = torch.cuda.mem_get_info(local)[0]
    need = (hi - lo) * per * 16 + m * 4096 * 4 + 3 * nq * 24 * 2
    per_fit = per
    if need > free_b * 0.92:   # the 16-B-per-seed layout holds 10^10 seeds only from 2 GPUs up: say so and shrink the buckets
        per_fit = int((free_b * 0.92 - m * 4096 * 4 - 3 * nq * 48) / ((hi - lo) * 16))
        log("rank %d: %d seeds per mask do not fit (%.0f GB needed, %.0f GB free): using %d" % (rank, per, need / 1e9, free_b / 1e9, per_fit))
    pf = torch.tensor([float(per_fit)], device="cuda", dtype=torch.float64)
    if dist:
        dist.all_reduce(pf, op=dist.ReduceOp.MIN)
    per_fit = int(pf.item())
    t0 = time.time()
    idx = lexicmap_b200.Index.synthetic(masks=m, per_mask=per_fit, seed=C5["seed"], mask_lo=lo, mask_hi=hi, device=local, with_values=False)
    torch.cuda.synchronize()
    log("rank %d: synthetic image masks [%d, %d) x %d seeds = %.1f GB in %.1fs" % (rank, lo, hi, per_fit, idx.info.image_bytes / 1e9, time.time() - t0))
    if dist:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    if a.warmup:
        idx.probe_bench(nq, iters=a.warmup)
    r = idx.probe_bench(nq, iters=a.steps)   # after one untimed lookup pass of its own
    sampler.finish()
    if a.dump_outputs and rank == 0:
        dump_arrays(a.dump_outputs, {"probe_" + k: [r[k]] for k in ("issued", "survivors", "hits", "sum_log2", "sum_hit_sectors", "sum_values", "steps", "entries")})

    t = torch.tensor([r["survivors"], r["issued"], r["hits"], r["sum_log2"], r["sum_hit_sectors"], r["sum_values"], r["kernel_ms"], r["kernel_ms_best"], r["regroup_ms"]], device="cuda", dtype=torch.float64)
    if dist:
        tm = t[6:].clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(t[:6], op=dist.ReduceOp.SUM)
        t[6:] = tm
    surv, issued, hits, slog, ssec, sval, kms, kbest, rms = (float(x) for x in t.tolist())
    step_ms = kms + rms   # a lookup step = regrouping pass (probes bucketed by mask) + lookup kernel
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return None
    peak, peak_src = hbm_peak()
    alg = probe_model_bytes(surv, slog, ssec, sval)
    per_gpu = alg / world / (kms * 1e-3) / 1e9
    out = {"metric": "seed lookups/s (prefix + suffix probes of 31-mers against the seed index)", "value": surv / (step_ms * 1e-3), "unit": "probes/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": step_ms,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
           "config": {"workload": "BASELINE.json configs[4]: %d query 31-mers (half stored keys mutated in their last 0-16 bases, half uniform), one prefix + one suffix probe each, vs a synthetic seed index of %d masks x %d seeds = %.2e seeds%s"
                                  % (nq, m, per_fit, m * per_fit, "" if per_fit == per else " (REDUCED from %d per mask: 16 B per seed, %d GPU(s))" % (per, world)),
                      "sharding": "index range-partitioned by mask over %d GPU(s); every probe goes to the GPU that owns its mask; no collective" % world, "seed": C5["seed"], "l2": "index shard (tens of GB) and the probe list (hundreds of MB) exceed the 126 MB L2"},
           "gpu_launches": 4 * (a.steps + a.warmup + 1) + 2, "probes_issued": issued, "probes_with_anchor": surv, "hit_records": hits,
           "roofline": {"bound": "hbm", "kernel": "k_probe_find2", "achieved": per_gpu, "peak": peak, "unit": "GB/s", "frac": per_gpu / peak, "traffic": None, "model": "SURVEY.md §8d per-probe bytes, per GPU (max kernel time over ranks)",
                        "algorithmic_bytes_per_step": alg, "bytes_per_probe": alg / max(surv, 1), "kernel_ms_per_step": kms, "kernel_ms_best": kbest, "regroup_ms_per_step": rms, "frac_with_regroup": alg / world / (step_ms * 1e-3) / 1e9 / peak, "mean_log2_steps": slog / max(surv, 1), "peak_source": peak_src,
                        "random_sector_ceiling": {"note": "measured rate of independent random 32-byte-sector reads over an 8-GB buffer (k_gather_bench): buckets of this index are MBs, so a probe's sectors still miss in L2 after the regrouping (which helps through the TLB)",
                                                  "sectors_per_s": gb["sectors_per_s"], "gbs_at_32B": gb["gbs_at_32B"], "frac_of_streaming_peak": gb["gbs_at_32B"] / peak}},
           "e2e": {"value": surv / (step_ms * 1e-3), "unit": "probes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": "device-resident microbenchmark: probes are generated on the GPU; the end-to-end numbers are the search configs'"},
           "cpu_baseline": None, "clocks": sampler.summary()}
    if dist:
        dist.destroy_process_group()
    return out


# ------------------------------------------------------------------------------------------------ reference arm (CPU port)
def run_reference(a):
    from oracle_binding import read_fasta
    threads = usable_cpus()[0]
    search_kw = {}
    note_extra = ""
    div = 1
    if a.config == "c2":
        idx_dir, qf = ensure_c2(0)
        ids, seqs = read_fasta(qf)
        workload = "%d synthetic %d-bp queries vs %d-genome synthetic index (%dx%dx%d bp), BASELINE.json configs[1]" % (C2["n_queries"], C2["query_len"], C2["families"] * C2["members"], C2["families"], C2["members"], C2["genome_len"])
        config = base_config(a, workload, {"queries_per_gpu": C2["n_queries"], "query_len": C2["query_len"], "genomes": C2["families"] * C2["members"], "masks": 20000,
                                           "sharding": "by query, index replicated" if a.gpus > 1 else "single GPU", "seeds": [C2["genome_seed"], C2["query_seed"]]})
    elif a.config == "c3":
        world = max(1, a.gpus)
        idx_dir = ensure_c3(0, world)
        ids, seqs = [], []
        parts = [read_fasta(qf)[1] for qf in c3_queries(world)]   # the whole batch: part 0 hits shard 0's genomes, the other parts only probe it (as on every GPU rank)
        per = min(len(x) for x in parts)
        seqs = [parts[p][i] for i in range(per) for p in range(world)]   # parts in turn: any prefix of the batch is a fair sample of the whole job
        ids = ["q%d" % i for i in range(len(seqs))]
        config = base_config(a, "BASELINE.json configs[2]: %d x %d-bp queries vs %d genomes, CPU port against shard 0 of %d" % (C3["n_queries"], C3["query_len"], C3["genomes"], world), {"genomes": C3["genomes"]})
        div = world
        note_extra = "; measured against shard 0 (1/%d of the genomes) and divided by %d" % (world, world)
    elif a.config == "c4":
        from conftest import DEMO_INDEX, GOLD
        idx_dir = DEMO_INDEX
        ids, seqs = read_fasta(os.path.join(GOLD, "demo_long_reads_subset.fasta.gz"))
        search_kw = dict(min_qcov_hsp=70.0, top_n_genomes=5, top_n_chains=1)
        config = base_config(a, "simulated ONT reads vs the reference's 15 demo genomes (BASELINE.json configs[3] on the demo index)", {"genomes": 15, "flags": search_kw})
    else:
        print(json.dumps({"impl": "reference", "unavailable": "the seed-lookup microbenchmark (c5) has no CPU arm: the reference's on-disk searcher is I/O bound by design (kv-searcher.go:366)"}))
        return
    vals = []
    for i in range(a.warmup + a.steps):
        bps, n, dt, nrows = cpu_port_throughput(idx_dir, seqs, threads, target_s=8.0, params=search_kw, whole=False)
        if i >= a.warmup:
            vals.append((bps / div, n, dt))
    bps = float(np.mean([v[0] for v in vals]))
    n, dt = vals[-1][1], float(np.mean([v[2] for v in vals]))
    print(json.dumps({"impl": "reference", "metric": "aligned query bp/s", "value": bps, "unit": "bp/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt * 1e3,
                      "higher_is_better": True, "scaling": "weak" if a.config != "c3" else "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic" if a.config != "c4" else "reference demo reads (simulated ONT)", "config": config,
                      "cpu_baseline": dict({"value": bps, "unit": "bp/s", "kind": "port", "sample": "%d of the %d queries per step (C++ port of the reference path; Go toolchain absent)%s" % (n, len(seqs), note_extra)}, **cpu_desc(threads)),
                      "e2e": {"value": bps, "unit": "bp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default=os.environ.get("LMG_BENCH_CONFIG", "c2"), choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if a.impl == "reference":
        if rank == 0:
            run_reference(a)
        return
    real_stdout = os.dup(1)
    os.dup2(2, 1)   # libraries (NCCL banner) must not pollute the one JSON line on stdout
    out = run_c5(a, rank, world, local) if a.config == "c5" else run_search(a, rank, world, local)
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    if out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
