"""Builds tests/golden/demo_refs_windows.tsv.gz and tests/golden/demo_long_reads_subset.fasta.gz, so that the demo tests run on
the reference's demo data without its 16 MB of genomes. usage: make_demo_fixture.py <LexicMap demo directory> (the one holding refs/).

The demo genomes are indexed here as they are, and the CPU oracle searches them with the test queries. The windows file keeps what those
searches and the reference's golden rows touch: the subject interval of every HSP, FLANK bases on each side (more than the 1,000-base
pseudo-alignment extension), plus every contig's name and length. tests/conftest.py::ensure_demo_index fills the rest of each contig with
seeded random bases, so coordinates, contig lengths and the index's total bases (hence e-values) stay those of the real genomes.

Long reads kept (from the sample written by make_long_read_fixture.py): every read of the reference's result overview, the shortest read
with an alignment longer than 50 kb, GENERAL_WFA_READ, and the N_CHEAP reads that need the least stored sequence among the others with at
least one row under the demo flags."""
import collections
import gzip
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import GOLD, _tools, read_tsv   # noqa: E402
from oracle_binding import Oracle, read_fasta   # noqa: E402
from test_oracle_cpu import LONG_READ_FLAGS   # noqa: E402

FLANK = 1200
N_CHEAP = 20
GENERAL_WFA_READ = "GCF_001457655.1_r115"   # measured on a B200: its 32-kb alignment leaves the register WFA kernels' window and takes k_wfa


def union(iv):
    out = []
    for a, b in sorted(iv):
        if out and a <= out[-1][1]:
            out[-1][1] = max(out[-1][1], b)
        else:
            out.append([a, b])
    return out


def main(demo):
    refs = os.path.join(demo, "refs")
    files = sorted(os.listdir(refs))
    with tempfile.TemporaryDirectory() as d:
        lst = os.path.join(d, "list")
        open(lst, "w").write("".join(os.path.join(refs, f) + "\n" for f in files))
        idx = os.path.join(d, "demo.lmi")
        subprocess.check_call([_tools(), "index", "--in-list", lst, "--out", idx], stderr=subprocess.DEVNULL)
        o = Oracle(idx)

        def hsps(seqs, **kw):
            rows, sid, _ = o.search(seqs, o.default_params(**kw), threads=os.cpu_count() or 8)
            return [(int(r["query"]), o.genome_name(r["genome"]), sid[i], int(r["tb"]), int(r["te"]), int(r["alen"])) for i, r in enumerate(rows)]
        iv = []
        for fa, kws in (("demo_q.gene.fasta", [dict(output_seq=1), dict(output_seq=1, top_n_genomes=2)]), ("demo_q.prophage.fasta", [dict(output_seq=1)])):
            for kw in kws:
                iv += [r[1:5] for r in hsps(read_fasta(os.path.join(GOLD, fa))[1], **kw)]
        for f in ("demo_q.gene.fasta.lexicmap.tsv", "demo_q.gene.top2_all.tsv", "demo_q.prophage.fasta.lexicmap.tsv", "demo_long_reads_readme_rows.tsv"):
            for r in read_tsv(os.path.join(GOLD, f)):
                a, b = sorted((int(r[14]) - 1, int(r[15]) - 1))
                iv.append((r[3], r[4], a, b))
        ids, seqs = read_fasta(os.path.join(GOLD, "demo_long_reads_sample.fasta.gz"))
        per = collections.defaultdict(list)
        for r in hsps(seqs, **LONG_READ_FLAGS):
            per[r[0]].append(r)
        readme = {r[0] for r in read_tsv(os.path.join(GOLD, "demo_long_reads_readme_rows.tsv"))}
        keep = {i for i, x in enumerate(ids) if x in readme}
        keep.add(min((len(seqs[q]), q) for q, rs in per.items() if max(r[5] for r in rs) > 50000)[1])
        cost = sorted((len(seqs[q]) + sum(r[4] - r[3] + 1 + 2 * FLANK for r in rs), q) for q, rs in per.items() if q not in keep)
        keep |= {q for _, q in cost[:N_CHEAP]}
        keep.add(ids.index(GENERAL_WFA_READ))
        keep = sorted(keep)
        for q in keep:
            iv += [r[1:5] for r in per[q]]
        o.close()

    win = collections.defaultdict(list)
    for g, s, a, b in iv:
        win[(g, s)].append((max(0, a - FLANK), b + FLANK))
    stored = 0
    with gzip.GzipFile(os.path.join(GOLD, "demo_refs_windows.tsv.gz"), "wb", mtime=0) as out:
        for f in files:
            g = f.split(".fa")[0]
            out.write(("G\t%s\n" % g).encode())
            for sid, seq in zip(*read_fasta(os.path.join(refs, f))):
                out.write(("C\t%s\t%d\n" % (sid, len(seq))).encode())
                for a, b in union(win.pop((g, sid), [])):
                    b = min(b, len(seq) - 1)
                    out.write(("W\t%d\t%s\n" % (a, seq[a:b + 1])).encode())
                    stored += b + 1 - a
    assert not win, "HSPs on contigs not in refs/: %s" % list(win)
    with gzip.GzipFile(os.path.join(GOLD, "demo_long_reads_subset.fasta.gz"), "wb", mtime=0) as f:
        for q in keep:
            f.write((">%s\n%s\n" % (ids[q], seqs[q])).encode())
    print("%d bases of genome windows; %d reads, %d bases" % (stored, len(keep), sum(len(seqs[q]) for q in keep)))


if __name__ == "__main__":
    main(sys.argv[1])
