"""GPU tests of the drop-in boundary and of the rows SURVEY.md §8 lists next to the kernels: the `lexicmap search` look-alike CLI (a19), the C
ABI under concurrent callers, split genomes / genome batches (a18), the on-device index ingest (§8f-2), genome shards and the synthetic
seed-lookup benchmark image (configs[4])."""
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLD, ROOT, read_tsv, tsv_key
from oracle_binding import Oracle, read_fasta

pytestmark = pytest.mark.gpu


def _same(a, b):
    (ra, sa, ca), (rb, sb, cb) = a, b
    assert len(ra) == len(rb), "row count differs: %d vs %d" % (len(ra), len(rb))
    for f in ra.dtype.names:
        if f not in ("cigar_off", "pad", "pad0"):
            assert np.array_equal(ra[f], rb[f]), "column %s differs" % f
    assert sa == sb and ca == cb


def _write_fasta(path, ids, seqs):
    with open(path, "w") as f:
        for i, s in zip(ids, seqs):
            f.write(">%s some description\n" % i)
            for x in range(0, len(s), 60):
                f.write(s[x:x + 60] + "\n")


def _cli():
    from lexicmap_b200 import build
    build.build_tools()
    return build.CLI


def test_cli_output_is_byte_identical_to_the_api_formatter(gpu_small, small_index, small_queries, tmp_path):
    """`lexicmap-gpu search -d ... -a` writes exactly the lines lexicmap_b200.api.Index.format_tsv produces from the same rows (which the CPU
    suite pins to the reference's golden files through the oracle's formatter); queries shorter than k are skipped as in search.go:571-575"""
    ids, seqs = small_queries
    qf = str(tmp_path / "q.fa")
    _write_fasta(qf, ids, seqs)
    for all_cols in (True, False):
        out = str(tmp_path / ("out%d.tsv" % all_cols))
        subprocess.check_call([_cli(), "search", "-d", small_index, qf, "-o", out, "--quiet"] + (["-a"] if all_cols else []))
        keep = [i for i, s in enumerate(seqs) if len(s) >= 31]
        rows, sid, cig = gpu_small.search([seqs[i] for i in keep], gpu_small.default_params(output_seq=int(all_cols)))
        want = gpu_small.format_tsv(rows, sid, [ids[i] for i in keep], [len(seqs[i]) for i in keep], cig if all_cols else None, gpu_small.last_align_text if all_cols else None)
        got = open(out).read().splitlines()
        assert got[0].split("\t")[:20] == "query qlen hits sgenome sseqid qcovGnm cls hsp qcovHSP alenHSP pident gaps qstart qend sstart send sstr slen evalue bitscore".split()
        assert got[1:] == want and len(want) > 50


def test_cli_on_the_demo_index_reproduces_reference_rows(demo_index, tmp_path):
    out = str(tmp_path / "gene.tsv")
    subprocess.check_call([_cli(), "search", "-d", demo_index, os.path.join(GOLD, "demo_q.gene.fasta"), "-o", out, "--quiet", "-j", "8"])
    mine = {tsv_key(f): f for f in read_tsv(out)}
    gold = {tsv_key(f): f for f in read_tsv(os.path.join(GOLD, "demo_q.gene.fasta.lexicmap.tsv"))}
    common = set(mine) & set(gold)
    assert len(common) >= 80 and not (set(mine) - set(gold))
    for kx in common:
        assert mine[kx][8:20] == gold[kx][8:20]
    # flags the GPU path does not implement are refused, not ignored
    r = subprocess.run([_cli(), "search", "-d", demo_index, "-w", os.path.join(GOLD, "demo_q.gene.fasta")], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode != 0 and "load-whole-seeds" in r.stderr


def test_measurement_switches_do_not_change_a_byte(demo_index, tmp_path):
    """the environment switches that exist for A/B measurements (probe regrouping, L2 eviction hints, 16-bit anchor starts, lookup stream priority,
    the 128- and 256-diagonal register WFA kernels) select other kernels or layouts, never other results: the `-a` TSV of the simulated ONT reads
    (wide-band alignments included) is byte-identical under each of them"""
    q = os.path.join(GOLD, "demo_long_reads_subset.fasta.gz")
    def run(tag, extra):
        out = str(tmp_path / (tag + ".tsv"))
        subprocess.check_call([_cli(), "search", "-d", demo_index, q, "-o", out, "--quiet", "-a"], env=dict(os.environ, **extra))
        return open(out, "rb").read()
    base = run("default", {})
    assert base.count(b"\n") > 40
    for name in ("LMG_NO_REGROUP", "LMG_L2_HINTS", "LMG_CSTART32", "LMG_NO_PRIO_LOOKUP", "LMG_NO_WFA_REG8", "LMG_NO_WFA_REG"):
        assert run(name, {name: "1"}) == base, name


def test_cli_reads_long_fastq_lines(gpu_small, small_index, small_queries, tmp_path):
    """a FASTQ record whose sequence line is longer than the 64-KB read buffer (ONT reads) must arrive whole"""
    ids, seqs = small_queries
    long_read = (seqs[0] + seqs[1] + seqs[2]) * 30          # ~72 kb on one line
    fq = str(tmp_path / "q.fq")
    with open(fq, "w") as f:
        f.write("@long1 x\n%s\n+\n%s\n@short1\n%s\n+\n%s\n" % (long_read, "I" * len(long_read), seqs[3], "I" * len(seqs[3])))
    out = str(tmp_path / "fq.tsv")
    subprocess.check_call([_cli(), "search", "-d", small_index, fq, "-o", out, "--quiet"])
    rows = read_tsv(out)
    assert {r[0] for r in rows} == {"long1", "short1"} and {int(r[1]) for r in rows if r[0] == "long1"} == {len(long_read)}


def test_two_host_threads_share_one_index(small_index, small_queries, tmp_path):
    ids, seqs = small_queries
    qf = str(tmp_path / "q.fa")
    _write_fasta(qf, ids, [s for s in seqs])
    exe = str(tmp_path / "capi_threads")
    lib = os.path.join(ROOT, "lexicmap_b200")
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", os.path.join(ROOT, "tests", "capi_threads.cpp"), "-o", exe, "-I", os.path.join(ROOT, "include"), "-L", lib, "-llexicmap_gpu", "-lpthread", "-Wl,-rpath," + lib])
    r = subprocess.run([exe, small_index, qf], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("ok"), (r.returncode, r.stdout, r.stderr)


def test_split_genomes_and_batches_match_oracle(split_index, split_queries):
    """genomes split into chunks (genomes.chunks.bin) over several genome batches: chunk merge, merged coverage, -Q, top-N order (a18)"""
    import lexicmap_b200
    from test_oracle_cpu import check_split_index_rows
    ids, seqs = split_queries
    g, o = lexicmap_b200.Index(split_index, device=0), Oracle(split_index)
    assert g.info.genome_batches >= 4
    for kw in (dict(output_seq=1), dict(min_qcov_genome=90.0), dict(top_n_genomes=3, output_seq=1), dict(top_n_genomes=2, top_n_chains=1, min_qcov_hsp=20.0)):
        res = g.search(seqs, g.default_params(**kw))
        _same(res, o.search(seqs, o.default_params(**kw)))
    rows, sid, cig = g.search(seqs, g.default_params())
    check_split_index_rows(split_index, rows, sid, ids, seqs, g.genome_name)
    assert g.anchors(seqs).tobytes() == o.anchors(seqs).tobytes()
    g.close()


def test_ingest_modes_and_reopen_give_the_same_image(small_index, gpu_small, small_queries):
    """the chunk files are decoded on the device in two passes; the raw bytes either stay on the device between the passes or are read again
    (LMG_INGEST_REREAD, the path taken by images that fill the GPU): both images answer identically, and so does a second open"""
    import lexicmap_b200
    ids, seqs = small_queries
    ref = gpu_small.search(seqs, gpu_small.default_params(output_seq=1))
    os.environ["LMG_INGEST_REREAD"] = "1"
    try:
        g = lexicmap_b200.Index(small_index, device=0)
    finally:
        del os.environ["LMG_INGEST_REREAD"]
    assert (g.info.seed_keys, g.info.seed_values, g.info.image_bytes) == (gpu_small.info.seed_keys, gpu_small.info.seed_values, gpu_small.info.image_bytes)
    _same(g.search(seqs, g.default_params(output_seq=1)), ref)
    assert g.anchors(seqs).tobytes() == gpu_small.anchors(seqs).tobytes()
    t = g.load_times()
    assert t["total_ms"] > 0 and t["seed_fill_ms"] > 0
    g.close()


def test_genome_shards_refuse_top_n_and_keep_first_value_flags(small_index, gpu_small, small_queries):
    import lexicmap_b200
    from lexicmap_b200.dist import merge_genome_shards
    ids, seqs = small_queries
    ref = gpu_small.search(seqs, gpu_small.default_params(output_seq=1))
    parts = []
    for sh in range(4):
        g = lexicmap_b200.Index(small_index, device=0, shard=sh, n_shards=4)
        parts.append(g.search(seqs, g.default_params(output_seq=1)))
        with pytest.raises(RuntimeError):
            g.search(seqs, g.default_params(top_n_genomes=2))
        g.close()
    _same(merge_genome_shards(parts), ref)


def test_total_bases_override_scales_evalues(small_index, small_queries):
    """a shard of a larger collection reports the e-values of the whole collection (lib-index-search.go:1918 uses the index's total bases)"""
    import lexicmap_b200
    ids, seqs = small_queries
    g = lexicmap_b200.Index(small_index, device=0)
    a = g.search(seqs, g.default_params(max_evalue=1e300))[0]
    g.set_total_bases(int(g.info.input_bases) * 8)
    b = g.search(seqs, g.default_params(max_evalue=1e300))[0]
    g.close()
    assert len(a) == len(b) and np.array_equal(a["bitscore"], b["bitscore"])
    nz = a["evalue"] > 0
    assert nz.any() and np.allclose(b["evalue"][nz], 8 * a["evalue"][nz], rtol=1e-12)


def test_synthetic_seed_image_probe_bench():
    """BASELINE.json configs[4] in miniature: stored keys mutated only beyond the 15-base minimum prefix must be found again"""
    import lexicmap_b200
    g = lexicmap_b200.Index.synthetic(masks=20000, per_mask=2000, seed=7)
    r = g.probe_bench(200000, iters=2)
    assert g.info.seed_keys == 20000 * 2000
    assert r["issued"] == 400000 and 0 < r["survivors"] <= r["issued"]
    assert r["hits"] >= 0.2 * 200000, r             # a key-derived query (half of them) finds its own key through the prefix probe when that key's first value is a forward one (half of those)
    assert r["sum_log2"] >= r["survivors"] and r["kernel_ms"] > 0
    with pytest.raises(RuntimeError):
        g.search(["ACGT" * 50])
    g.close()
    # range partition by mask: the two halves issue disjoint probe sets that add up to the whole
    a = lexicmap_b200.Index.synthetic(masks=20000, per_mask=2000, seed=7, mask_lo=0, mask_hi=10000)
    b = lexicmap_b200.Index.synthetic(masks=20000, per_mask=2000, seed=7, mask_lo=10000, mask_hi=20000)
    ra, rb = a.probe_bench(200000, iters=1), b.probe_bench(200000, iters=1)
    a.close()
    b.close()
    assert ra["issued"] + rb["issued"] == r["issued"] and ra["survivors"] + rb["survivors"] == r["survivors"] and ra["hits"] + rb["hits"] == r["hits"]
