"""GPU parity on the reference's own demo data: the CUDA path (through the C ABI) against the CPU oracle — bit for bit — AND against the
reference's golden output rows (tests/golden/, copied from the reference's demo/). The index is tests/data/demo.lmi: the reference's 15 demo
genomes (the windows stored in tests/golden/, seeded filler elsewhere) indexed by this repo's writer with the reference's default options
(20,000 masks, seed-desert filling). Covers BASELINE.json configs[0] (gene queries), the 33.6-kb prophage query and configs[3]
(simulated ONT reads, two of them beyond the fast WFA kernel's 32,000-base limit)."""
import os

import numpy as np
import pytest

from conftest import GOLD, read_tsv, tsv_key
from oracle_binding import Oracle, read_fasta

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def demo(demo_index):
    import lexicmap_b200
    g = lexicmap_b200.Index(demo_index, device=0)
    yield g, Oracle(demo_index)
    g.close()


def _same(a, b):
    (ra, sa, ca), (rb, sb, cb) = a, b
    assert len(ra) == len(rb), "row count differs: gpu %d oracle %d" % (len(ra), len(rb))
    for f in ra.dtype.names:
        if f not in ("cigar_off", "pad", "pad0"):
            assert np.array_equal(ra[f], rb[f]), "column %s differs" % f
    assert sa == sb and ca == cb


def _tsv(g, res, ids, seqs, all_cols=False):
    rows, sid, cig = res
    lines = g.format_tsv(rows, sid, ids, [len(s) for s in seqs], cig if all_cols else None, g.last_align_text if all_cols else None)
    return {tsv_key(l.split("\t")): l.split("\t") for l in lines}


def test_gene_queries_match_oracle_and_reference_rows(demo):
    g, o = demo
    ids, seqs = read_fasta(os.path.join(GOLD, "demo_q.gene.fasta"))
    res = g.search(seqs, g.default_params(output_seq=1))
    _same(res, o.search(seqs, o.default_params(output_seq=1), threads=8))
    assert g.last_align_text == o.last_align_text
    mm = _tsv(g, res, ids, seqs, all_cols=True)
    gm = {tsv_key(f): f for f in read_tsv(os.path.join(GOLD, "demo_q.gene.fasta.lexicmap.tsv"))}
    common = set(gm) & set(mm)
    assert len(gm) == 84 and len(common) >= 80 and not (set(mm) - set(gm))
    for kx in common:
        assert gm[kx][8:20] == mm[kx][8:20], (gm[kx], mm[kx])            # alenHSP pident gaps qstart qend sstart send sstr slen evalue bitscore
    n = 0
    for f in read_tsv(os.path.join(GOLD, "demo_q.gene.top2_all.tsv")):
        if tsv_key(f) in mm:
            assert mm[tsv_key(f)][20:24] == f[20:24], "CIGAR / qseq / sseq / align differ from the reference's -a output"
            n += 1
    assert n == 14


def test_prophage_query_matches_oracle_and_reference_rows(demo):
    g, o = demo
    ids, seqs = read_fasta(os.path.join(GOLD, "demo_q.prophage.fasta"))
    res = g.search(seqs, g.default_params(output_seq=1))
    _same(res, o.search(seqs, o.default_params(output_seq=1), threads=8))
    mm = _tsv(g, res, ids, seqs)
    gm = {tsv_key(f): f for f in read_tsv(os.path.join(GOLD, "demo_q.prophage.fasta.lexicmap.tsv"))}
    common = set(gm) & set(mm)
    assert len(common) >= 5
    whole = {f[3] for f in gm.values()} - {gm[kx][3] for kx in set(gm) - common}   # qcovGnm where every reference HSP of the genome is reproduced (test_oracle_cpu)
    for kx in common:
        assert gm[kx][8:20] == mm[kx][8:20] and (gm[kx][3] not in whole or gm[kx][5] == mm[kx][5]), (gm[kx], mm[kx])
    assert {int(gm[kx][9]) for kx in common} >= {9371, 6942, 5941, 820}


@pytest.fixture(scope="module")
def long_reads():
    return read_fasta(os.path.join(GOLD, "demo_long_reads_subset.fasta.gz"))


def test_long_reads_match_oracle_and_reference_rows(demo, long_reads):
    """the reference's own long-read demo (demo/README.md:365-419): --min-qcov-per-hsp 70 --top-n-genomes 5 --top-n-chains 1"""
    g, o = demo
    ids, seqs = long_reads
    assert sum(len(s) > 32000 for s in seqs) >= 1 and max(len(s) for s in seqs) > 60000
    kw = dict(min_qcov_hsp=70.0, top_n_genomes=5, top_n_chains=1, output_seq=1)
    res = g.search(seqs, g.default_params(**kw))
    _same(res, o.search(seqs, o.default_params(**kw), threads=os.cpu_count() or 8))
    assert int(g.timing()[1][11]) > 0, "some alignments must have taken the general WFA kernel (sequences >= 32,000 bases)"
    mm = _tsv(g, res, ids, seqs)
    gold = read_tsv(os.path.join(GOLD, "demo_long_reads_readme_rows.tsv"))
    for f in gold:
        assert tsv_key(f) in mm, f
        assert mm[tsv_key(f)][3:20] == f[3:20], (f, mm[tsv_key(f)])
    assert len(res[0]) > 30 and int(res[0]["alen"].max()) > 50000


def test_long_reads_default_flags_match_oracle(demo, long_reads):
    """no top-N limits: every candidate genome and chain of a read is pseudo-aligned and aligned (many short, divergent HSPs)"""
    g, o = demo
    ids, seqs = long_reads
    for lanes in (1, 3):
        res = g.search(seqs, g.default_params(output_seq=1, lanes=lanes))
        _same(res, o.search(seqs, o.default_params(output_seq=1), threads=os.cpu_count() or 8))
