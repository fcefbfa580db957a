"""CPU suite (-m "not gpu"): pins the oracle against the reference's own known-answer tests and golden outputs, checks the
product's host-side format code, and that the C-ABI library exports everything include/lexicmap_gpu.h declares."""
import os
import random
import re
import subprocess

import numpy as np
import pytest

from conftest import GOLD, ROOT, _tools, make_index, read_chunk_groups, read_tsv, tsv_key
from oracle_binding import Oracle, read_fasta, format_tsv



# ------------------------------------------------------------------ reference KAT: kv/kv-data_test.go:30-283
def test_kv_known_answer(tmp_path):
    f = str(tmp_path / "t.kv")
    subprocess.check_call([_tools(), "kat", "--out", f])
    o = Oracle(None)
    o.open_kv(f)
    k, lp = 5, 2
    prefix = 0b0111 << ((k - lp) << 1)
    n = 1 << ((k - lp) << 1)
    n_masks = 1 << lp
    for p in (4, 5):
        for i in range(1, n - 1):
            tot, exact = 0, False
            for j in range(n_masks):
                cnt, lens, vals = o.kv_search(j, prefix | i, p, check_flag=False)
                tot += cnt
                for L, v in zip(lens, vals):
                    if L == k and v == i:
                        exact = True
            assert tot == n_masks * (1 << ((k - p) << 1)), (p, i, tot)
            assert exact


def test_product_kv_decoder_on_kat(tmp_path):
    """the product's chunk decoder (used to build the GPU image) reads back exactly what the KAT wrote"""
    f = str(tmp_path / "t.kv")
    subprocess.check_call([_tools(), "kat", "--out", f])
    out = subprocess.check_output([_tools(), "kv-dump", "--file", f], text=True).splitlines()
    assert out[0].startswith("k=5 mask_offset=0 chunk_size=4 mask_prefix=2 anchor_prefix=2 use7=1")
    keys = [l.split("\t") for l in out if l.startswith("K")]
    assert len(keys) == 4 * 64
    prefix = 0b0111 << 6
    for m in range(4):
        mk = [(int(x[2]), int(x[3])) for x in keys if int(x[1]) == m]
        assert mk == [(prefix | i, i) for i in range(64)]
    anchors = [l.split("\t") for l in out if l.startswith("A")]
    # anchor = bases [2,4) of the 5-mer; 16 anchors per mask, anchor a starts at key index 4*a
    for m in range(4):
        am = {int(x[2]): int(x[3]) for x in anchors if int(x[1]) == m}
        assert am == {a: 4 * a for a in range(16)}


def test_varint_gb_roundtrip():
    out = subprocess.check_output([_tools(), "varint-test", "--seed", "42"], text=True)
    assert "varint mismatches: 0" in out


# ------------------------------------------------------------------ tree.Search semantics (tree/tree_test.go; tree.go:441-527)
def _lcp(a, b, k):
    for i in range(k):
        sh = 2 * (k - 1 - i)
        if (a >> sh) & 3 != (b >> sh) & 3:
            return i
    return k


def test_tree_search_is_prefix_range_plus_documented_quirk():
    o = Oracle(None)
    rnd = random.Random(1)
    k = 21
    quirk = 0
    for trial in range(30):
        n = rnd.choice([1, 2, 100, 2000])
        keys = sorted({rnd.getrandbits(2 * k) for _ in range(n)} | {rnd.getrandbits(2 * 6) << (2 * (k - 6)) for _ in range(n // 10)})
        for _ in range(300):
            q = rnd.choice(keys) ^ (rnd.getrandbits(2 * rnd.randint(0, k)))
            if rnd.random() < 0.3:   # poly-A stretches trigger the uint8-wrap quirk
                pos = rnd.randint(2, 12)
                q &= ~(((1 << (2 * 6)) - 1) << (2 * (k - pos - 6)))
            p = rnd.randint(1, 14)
            ok, lo, hi = o.tree_search(keys, k, q, p)
            want = [i for i, x in enumerate(keys) if _lcp(x, q, k) >= p]
            got = list(range(lo, hi)) if ok else []
            if want:
                assert got == want
            elif got:   # spurious hits only when the query's bases [.., p) that still had to match are all A (tree.go:498-501)
                quirk += 1
                assert ((q >> (2 * (k - p))) & 0xF) == 0
    assert quirk > 0, "the quirk path should be exercised"


def test_dust_matches_definition():
    o = Oracle(None)
    rnd = random.Random(3)
    for _ in range(2000):
        kmer = rnd.getrandbits(62) if rnd.random() < 0.5 else int("".join(rnd.choice(["00", "01"]) for _ in range(31)), 2)
        cnt = {}
        for i in range(30):
            w = (kmer >> (2 * i)) & 63
            cnt[w] = cnt.get(w, 0) + 1
        want = sum(c * (c - 1) // 2 for c in cnt.values()) > 50
        assert bool(o.lib.lmo_dust(kmer, 31)) == want


# ------------------------------------------------------------------ genome store round trip (genome/genome_test.go)
def test_genome_subseq_roundtrip(tmp_path):
    refs = str(tmp_path / "refs")
    subprocess.check_call([_tools(), "synth-fasta", "--synth", "2,2,12000,5,3", "--out", refs])
    idx = make_index(tmp_path, "rt", "2,2,12000,5,3", chunks=2)
    o = Oracle(idx)
    rnd = random.Random(2)
    for gi, name in enumerate(sorted(os.listdir(refs))):
        ids, seqs = read_fasta(os.path.join(refs, name))
        concat = ("A" * 1000).join(seqs)
        assert o.genome_name(gi) == name[:-3]
        for _ in range(50):
            a = rnd.randrange(len(concat))
            b = min(len(concat) - 1, a + rnd.randrange(1, 500))
            assert o.subseq(gi, a, b) == concat[a:b + 1]
        assert o.subseq(gi, len(concat) - 10, len(concat) + 50) == concat[-10:]   # clamp at the genome end (genome.go:951-953)


# ------------------------------------------------------------------ golden demo outputs of the reference (v0.10.0)
# The demo index (tests/data/demo.lmi) is written by this repo's writer with the reference's default options (20,000 masks, seed-desert
# filling) from the reference's 15 demo genomes (their stored windows, conftest.write_demo_refs). Masks differ from the reference's (Go math/rand stream), so a few low-identity rows of the
# reference may be missing and `hits` may differ; every row found by both must agree in columns 9-20 (alenHSP ... bitscore) and qcovGnm.
def _demo_rows(o, fasta, **kw):
    ids, seqs = read_fasta(os.path.join(GOLD, fasta))
    rows, sid, cig = o.search(seqs, o.default_params(**kw), threads=8)
    lines = format_tsv(rows, sid, ids, [len(s) for s in seqs], o.genome_name, cig if kw.get("output_seq") else None, o.last_align_text if kw.get("output_seq") else None)
    return {tsv_key(l.split("\t")): l.split("\t") for l in lines}


def test_oracle_reproduces_reference_demo_rows(demo_index):
    """End-to-end pin of stages 1-5 incl. the two absent Go modules (lexichash, wfa): rows of demo/q.gene.fasta.lexicmap.tsv and the
    CIGAR / qseq / sseq / align columns of demo/q.gene.fasta.lexicmap_top-2-genomes_all.tsv."""
    o = Oracle(demo_index)
    mm = _demo_rows(o, "demo_q.gene.fasta", output_seq=1)
    gold = read_tsv(os.path.join(GOLD, "demo_q.gene.fasta.lexicmap.tsv"))
    gm = {tsv_key(f): f for f in gold}
    common = set(gm) & set(mm)
    assert len(gold) == 84 and len(common) >= 80, (len(gold), len(common))
    assert not (set(mm) - set(gm)), "rows not in the reference output"
    for kx in common:
        assert gm[kx][8:20] == mm[kx][8:20], (gm[kx], mm[kx])
    n = 0
    for f in read_tsv(os.path.join(GOLD, "demo_q.gene.top2_all.tsv")):
        if tsv_key(f) in mm:
            assert mm[tsv_key(f)][20] == f[20], "CIGAR differs"
            assert mm[tsv_key(f)][21:24] == f[21:24], "qseq / sseq / align text differs"   # cigar.AlignmentText of the absent wfa module, pinned by the golden -a rows
            n += 1
    assert n == 14


def test_oracle_reproduces_reference_prophage_rows(demo_index):
    """Long-query pin: demo/q.prophage.fasta (33.6 kb). With the writer's restatement of seed-desert filling (lib-index-build.go:1086-1413,
    the reference's default) the oracle reproduces the reference's long HSPs exactly — alignments of 9,371 / 6,942 / 5,941 / 2,983 / 820
    columns incl. gap columns, coordinates, pident, bit score, e-value and the genome coverage — which pins chaining over many seeds,
    windows >= 10 kb (minimum prefix 13) and WFA-adaptive on long alignments. Rows that depend on seeds of two low-identity genomes differ
    (other masks than the reference's). The 2,983-column HSP (and with it the genome coverage of GCF_003697165.2) also depends on which
    k-mers of its window win their masks against the whole genome: the demo index keeps only windows of the genomes (conftest.write_demo_refs)
    and extends that HSP by 38 columns, so qcovGnm is compared for the genomes whose reference HSPs are all reproduced."""
    o = Oracle(demo_index)
    mm = _demo_rows(o, "demo_q.prophage.fasta")
    gold = read_tsv(os.path.join(GOLD, "demo_q.prophage.fasta.lexicmap.tsv"))
    gm = {tsv_key(f): f for f in gold}
    common = set(gm) & set(mm)
    assert len(gold) == 9 and len(common) >= 5
    whole = {f[3] for f in gold} - {gm[kx][3] for kx in set(gm) - common}
    for kx in common:
        assert gm[kx][8:20] == mm[kx][8:20] and (gm[kx][3] not in whole or gm[kx][5] == mm[kx][5]), (gm[kx], mm[kx])     # columns 9-20 and qcovGnm
    assert {int(gm[kx][9]) for kx in common} >= {9371, 6942, 5941, 820}


LONG_READ_FLAGS = dict(min_qcov_hsp=70.0, top_n_genomes=5, top_n_chains=1)   # demo/README.md:365-368


def test_oracle_reproduces_reference_long_read_rows(demo_index):
    """BASELINE.json configs[3] pin: the ten rows the reference prints for demo/q.long-reads.fasta.gz (demo/README.md:410-419; simulated
    ONT reads of 2-20 kb, alignments of 2,101-20,481 columns with up to 307 gap columns) are reproduced in every column but `hits`
    (other masks find further low-identity genomes). Pins WFA-adaptive and the backtrace tie-breaking on noisy long alignments."""
    o = Oracle(demo_index)
    mm = _demo_rows(o, "demo_long_reads_subset.fasta.gz", **LONG_READ_FLAGS)
    gold = read_tsv(os.path.join(GOLD, "demo_long_reads_readme_rows.tsv"))
    assert len(gold) == 10
    for f in gold:
        assert tsv_key(f) in mm, f
        g = mm[tsv_key(f)]
        assert g[:2] == f[:2] and g[3:20] == f[3:20], (f, g)
    assert len(mm) > 30


# ------------------------------------------------------------------ regression pin on a deterministic synthetic fixture
def test_oracle_small_fixture_regression(oracle_small, small_queries):
    ids, seqs = small_queries
    rows, sid, cig = oracle_small.search(seqs, oracle_small.default_params(output_seq=1))
    mine = format_tsv(rows, sid, ids, [len(s) for s in seqs], oracle_small.genome_name, cig)
    # alignment text is consistent with the CIGAR (incl. gap columns, which the reference's golden -a rows do not contain)
    import re
    for c, (qs, ts, al), r in zip(cig, oracle_small.last_align_text, rows):
        assert len(qs) == len(ts) == len(al) == r["alen"]
        pos = 0
        for n_, op in re.findall(r"(\d+)([MXID])", c):
            n_ = int(n_)
            seg_q, seg_t, seg_a = qs[pos:pos + n_], ts[pos:pos + n_], al[pos:pos + n_]
            if op == "M":
                assert seg_a == "|" * n_ and seg_q.upper() == seg_t
            elif op == "X":
                assert seg_a == " " * n_ and all(a.upper() != b for a, b in zip(seg_q, seg_t))
            elif op == "I":
                assert seg_t == "-" * n_ and "-" not in seg_q and seg_a == " " * n_
            else:
                assert seg_q == "-" * n_ and "-" not in seg_t and seg_a == " " * n_
            pos += n_
        assert pos == r["alen"] and qs.replace("-", "").upper() == seqs[r["query"]][r["qb"]:r["qe"] + 1].upper()
    gold = os.path.join(GOLD, "small_expected.tsv")
    if os.environ.get("LMG_REGEN_GOLDEN"):
        open(gold, "w").write("\n".join(mine) + "\n")
    assert mine == open(gold).read().splitlines()


def check_split_index_rows(index_dir, rows, sid, ids, seqs, genome_name):
    """properties of a search against an index with split genomes and several genome batches (lib-index-search.go:2797-2913): the chunks of a
    genome are merged into one result (one name per query, `hits` = distinct names), qcovGnm is the union coverage over all of the genome's
    HSPs, cls/hsp count through the merged genome, chunk fields agree with genomes.chunks.bin."""
    groups = read_chunk_groups(index_dir)
    assert len(groups) >= 3 and all(len(g) >= 2 for g in groups)
    assert any((b >> 17) > 0 for g in groups for b in g), "some chunks live in genome batches > 0"
    merged = 0
    for q in np.unique(rows["query"]):
        r = rows[rows["query"] == q]
        names = [genome_name(g) for g in r["genome"]]
        order = list(dict.fromkeys(names))
        assert [k for k, _ in __import__("itertools").groupby(names)] == order, "a genome's rows are contiguous: chunks were merged"
        assert np.all(r["hits"] == len(order))
        for nm in order:
            rr = r[[n_ == nm for n_ in names]]
            cov = np.zeros(len(seqs[q]), bool)
            for a, b in zip(rr["qb"], rr["qe"]):
                cov[a:b + 1] = True
            assert abs(min(100.0, cov.sum() / len(seqs[q]) * 100) - rr["qcov_gnm"][0]) < 1e-9 and np.all(rr["qcov_gnm"] == rr["qcov_gnm"][0])
            assert list(rr["hsp"]) == list(range(1, len(rr) + 1)) and rr["cls"][0] == 1 and np.all(np.diff(rr["cls"]) >= 0)
            if len(set(zip(rr["chunk_idx"], rr["n_chunks"]))) > 1:
                merged += 1
            assert np.all(rr["chunk_idx"] < rr["n_chunks"])
    assert merged > 0, "at least one query hits two chunks of the same genome"


def test_split_genomes_and_batches(split_index, small_index, split_queries):
    ids, seqs = split_queries
    o = Oracle(split_index)
    info = open(os.path.join(split_index, "info.toml")).read()
    assert int(re.search(r"genome-batches\s*=\s*(\d+)", info).group(1)) >= 4 and int(re.search(r"\ngenomes\s*=\s*(\d+)", info).group(1)) > 16
    rows, sid, cig = o.search(seqs, o.default_params(output_seq=1))
    check_split_index_rows(split_index, rows, sid, ids, seqs, o.genome_name)
    # same genomes unsplit: every query that is found there is found here too
    o2 = Oracle(small_index)
    rows2, _, _ = o2.search(seqs, o2.default_params())
    assert set(np.unique(rows2["query"])) <= set(np.unique(rows["query"]))
    # -Q is applied to the merged coverage
    rq, _, _ = o.search(seqs, o.default_params(min_qcov_genome=90.0))
    assert len(rq) < len(rows) and np.all(rq["qcov_gnm"] >= 90.0)
    chim = [i for i, x in enumerate(ids) if x.startswith("chimera")]
    assert set(chim) <= set(np.unique(rq["query"]).tolist()), "each half covers 50 % of a chimera: it passes -Q 90 only through the merged coverage"


def test_mask_fast_equals_bruteforce_definition(oracle_small, small_queries):
    ids, seqs = small_queries
    a = oracle_small.mask(seqs[:2] + seqs[-3:], 20000)
    b = oracle_small.mask(seqs[:2] + seqs[-3:], 20000, bruteforce=True)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


# ------------------------------------------------------------------ the boundary
def test_capi_exports_every_declared_symbol():
    import ctypes
    from lexicmap_b200 import build
    lib = ctypes.CDLL(build.build_gpu_lib())
    hdr = open(os.path.join(ROOT, "include", "lexicmap_gpu.h")).read()
    names = set(re.findall(r"\b(lmg_[a-z_]+)\s*\(", hdr))
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), "missing export " + n


def test_no_gpu_means_loud_failure(small_index):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import lexicmap_b200
    with pytest.raises(RuntimeError):
        lexicmap_b200.Index(small_index)


def test_tsv_number_formats():
    # Go's %.3f / %.2e == C printf == Python % (two-digit exponent), search.go:492-518
    assert "%.2e" % 5.17090374e-304 == "5.17e-304" and "%.2e" % 0.0 == "0.00e+00" and "%.2e" % 1.72e-43 == "1.72e-43" and "%.3f" % 99.8054 == "99.805"


def test_all_columns_pool_layout_and_formatters(oracle_small, small_queries):
    """`-a` output: the string pool entry of a row is cigar | qseq | sseq | align; the product-side splitter (lexicmap_b200.api) recovers the
    same texts as the oracle binding, and both TSV formatters write identical 24-column lines (search.go:505-518)."""
    from lexicmap_b200.api import split_align_text
    ids, seqs = small_queries
    rows, sid, cig = oracle_small.search(seqs, oracle_small.default_params(output_seq=1))
    texts = oracle_small.last_align_text
    pool = b"".join((c + q + s + a).encode() for c, (q, s, a) in zip(cig, texts))
    r2 = rows.copy()
    off = 0
    for i in range(len(r2)):
        r2["cigar_off"][i] = off
        off += int(r2["cigar_len"][i]) + 3 * int(r2["alen"][i])
    assert split_align_text(r2, pool) == texts
    assert split_align_text(rows[:0], b"") is None
    lines = format_tsv(rows, sid, ids, [len(s) for s in seqs], oracle_small.genome_name, cig, texts)

    class _Fake:   # the product formatter only needs genome_name
        genome_name = staticmethod(oracle_small.genome_name)
    import lexicmap_b200.api as api
    assert api.Index.format_tsv(_Fake, rows, sid, ids, [len(s) for s in seqs], cig, texts) == lines
    f = lines[0].split("\t")
    assert len(f) == 24 and len(f[21]) == len(f[22]) == len(f[23]) == int(f[9])


def test_desert_filling_closes_seed_gaps(tmp_path):
    """index writer, seed-desert filling (on by default; lib-index-build.go:1086-1413): first-round seeds leave gaps of >= 100 bases between consecutive seed
    positions; after filling, gaps above max_desert + seed_dist survive only next to contig-interval regions, the first-round seeds are
    all still there, and every extra seed also has its base-reversed copy (reverse flag 1)."""
    import glob
    tools = _tools()

    def seed_positions(idx):
        fwd, rev = {}, {}
        for f in sorted(glob.glob(os.path.join(idx, "seeds", "chunk_*.bin"))):
            for line in subprocess.check_output([tools, "kv-dump", "--file", f], text=True).splitlines():
                p = line.split("\t")
                if p[0] != "K":
                    continue
                for v in p[3:]:
                    v = int(v)
                    (rev if v & 1 else fwd).setdefault((v >> 30) & 131071, set()).add((v >> 2) & ((1 << 28) - 1))
        return fwd, rev
    a = str(tmp_path / "plain.lmi")
    b = str(tmp_path / "filled.lmi")
    # 2,048 masks over 200-kb genomes: ~100 bases between first-round seeds on average, so deserts are common (20,000 masks would leave none here)
    subprocess.check_call([tools, "index", "--synth", "2,2,200000,5,3", "--out", a, "--chunks", "4", "--masks", "2048", "--no-fill-deserts"], stderr=subprocess.DEVNULL)
    subprocess.check_call([tools, "index", "--synth", "2,2,200000,5,3", "--out", b, "--chunks", "4", "--masks", "2048"], stderr=subprocess.DEVNULL)
    (fa, ra), (fb, rb) = seed_positions(a), seed_positions(b)
    assert set(fa) == set(fb)
    for g in fa:
        assert fa[g] <= fb[g] and fb[g] == rb[g] and fa[g] == ra[g]
        pa, pb = sorted(fa[g]), sorted(fb[g])
        gaps_a = [y - x for x, y in zip(pa, pa[1:])]
        gaps_b = [y - x for x, y in zip(pb, pb[1:])]
        assert max(gaps_a) >= 300                       # first round alone leaves deserts
        big = [d for d in gaps_b if d > 150]
        assert len(big) <= 4 and all(d >= 1000 for d in big if d > 400)   # only the 1000-bp contig intervals (<= 2 per genome) stay wide
        assert len(pb) > 1.5 * len(pa)
    assert "max-seed-dist = 100" in open(os.path.join(b, "info.toml")).read().replace('"', "") or "100" in open(os.path.join(b, "info.toml")).read()


def test_no_statement_hides_behind_a_line_comment():
    """the CUDA sources use long lines; a `//` comment in the middle of one silently disables whatever follows it (it happened twice: a
    kernel launch vanished without a compile error). Nothing that looks like a launch, a checked call or a declaration / statement after a semicolon may follow a `//` on its line."""
    import glob
    bad = []
    for f in glob.glob(os.path.join(ROOT, "lexicmap_b200", "csrc", "*")) + glob.glob(os.path.join(ROOT, "oracle", "*.?pp")):
        for n, line in enumerate(open(f, errors="replace"), 1):
            code, in_str, i = line, False, 0
            while i < len(code) - 1:
                c = code[i]
                if c == '"' and (i == 0 or code[i - 1] != "\\"):
                    in_str = not in_str
                if not in_str and code[i:i + 2] == "//":
                    rest = code[i + 2:]
                    if re.search(r"<<<[^>]*>>>|CUDA_CHECK\(|KERNEL_CHECK\(\)", rest) or re.search(r";\s*(u8|u16|u32|u64|i32|i64|int|bool|float|double|const|auto|std::|cuda[A-Z]\w*|CubTemp|DBuf|size_t|return|if \(|for \(|while \()\b", rest):
                        bad.append("%s:%d" % (os.path.basename(f), n))
                    break
                i += 1
    assert not bad, "code after a line comment: " + ", ".join(bad)
