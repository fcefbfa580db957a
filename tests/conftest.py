import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _tools():
    from lexicmap_b200 import build
    return build.build_tools()


def make_index(tmp, name, synth, masks=20000, chunks=4, extra=()):
    out = os.path.join(str(tmp), name + ".lmi")
    if not os.path.exists(os.path.join(out, "info.toml")):
        subprocess.check_call([_tools(), "index", "--synth", synth, "--out", out, "--masks", str(masks), "--chunks", str(chunks), *extra], stderr=subprocess.DEVNULL)
    return out


def make_queries(tmp, index, name, n, length, seed=20260925, max_sub=0.10, max_indel=0.01):
    out = os.path.join(str(tmp), name + ".fa")
    subprocess.check_call([_tools(), "synth-queries", "--index", index, "--n", str(n), "--len", str(length), "--seed", str(seed), "--out", out,
                           "--max-sub", str(max_sub), "--max-indel", str(max_indel)])
    return out


DEMO_INDEX = os.path.join(ROOT, "tests", "data", "demo.lmi")
GOLD = os.path.join(ROOT, "tests", "golden")
DEMO_FILL_SEED = 20261017


def write_demo_refs(out_dir):
    """the reference's 15 demo genomes as the demo tests see them (tests/golden/demo_refs_windows.tsv.gz, made by
    scripts/make_demo_fixture.py): every contig at its real length, the real bases in the stored windows around the HSPs the tests check,
    seeded random bases everywhere else (one PCG64 stream over all contigs, so no two contigs share filler). Returns the FASTA paths."""
    import gzip
    import numpy as np
    rng = np.random.PCG64(DEMO_FILL_SEED)   # the raw bit stream, which numpy keeps stable across versions
    acgt = np.frombuffer(b"ACGT", np.uint8)

    def filler(n):
        b = rng.random_raw(n // 32 + 1).view(np.uint8)
        return acgt[np.stack([b & 3, (b >> 2) & 3, (b >> 4) & 3, b >> 6], 1).reshape(-1)[:n]]
    paths, f, seq = [], None, None

    def flush():
        if seq is not None:
            f.write(b"%s\n" % seq.tobytes())
    with gzip.open(os.path.join(GOLD, "demo_refs_windows.tsv.gz"), "rt") as src:
        for line in src:
            t = line.rstrip("\n").split("\t")
            if t[0] == "G":
                flush()
                seq = None
                if f:
                    f.close()
                paths.append(os.path.join(out_dir, t[1] + ".fa"))
                f = open(paths[-1], "wb")
            elif t[0] == "C":
                flush()
                f.write(b">%s\n" % t[1].encode())
                seq = filler(int(t[2]))
            else:
                a = int(t[1])
                seq[a:a + len(t[2])] = np.frombuffer(t[2].encode(), np.uint8)
    flush()
    f.close()
    return paths


def ensure_demo_index():
    """index of the demo genomes (write_demo_refs) written by this repo's writer with the reference's default options (20,000 masks,
    seed-desert filling). Built once, by __graft_entry__.build() or by the first test that needs it; tests/data/ is git-ignored."""
    if os.path.exists(os.path.join(DEMO_INDEX, "info.toml")):
        return DEMO_INDEX
    import shutil
    import tempfile
    os.makedirs(os.path.dirname(DEMO_INDEX), exist_ok=True)
    tmp = DEMO_INDEX + ".tmp%d" % os.getpid()
    with tempfile.TemporaryDirectory() as d:
        lst = os.path.join(d, "list")
        with open(lst, "w") as f:
            f.write("".join(p + "\n" for p in write_demo_refs(d)))
        subprocess.check_call([_tools(), "index", "--in-list", lst, "--out", tmp], stderr=subprocess.DEVNULL)
    if os.path.isdir(DEMO_INDEX):
        shutil.rmtree(DEMO_INDEX)
    os.rename(tmp, DEMO_INDEX)
    return DEMO_INDEX


@pytest.fixture(scope="session")
def demo_index():
    return ensure_demo_index()


def tsv_key(f):
    """identity of an output row across implementations with different masks: query, genome, sequence, coordinates, strand"""
    return (f[0], f[3], f[4], f[12], f[13], f[14], f[15], f[16])


def read_tsv(path):
    return [l.rstrip("\n").split("\t") for l in open(path)][1:]


@pytest.fixture(scope="session")
def workdir(tmp_path_factory):
    return tmp_path_factory.mktemp("lmi")


@pytest.fixture(scope="session")
def small_index(workdir):
    """4 families x 4 members x 40 kb, multi-contig; 20,000 masks (the reference default)."""
    return make_index(workdir, "small", "4,4,40000,42,3")


@pytest.fixture(scope="session")
def small_queries(workdir, small_index):
    from oracle_binding import read_fasta
    ids, seqs = read_fasta(make_queries(workdir, small_index, "small_q", 24, 800))
    # edge cases: shorter than k, exactly k, poly-A, lower case, with N
    seqs += ["ACGTACGTAC", seqs[0][:31], "A" * 200, seqs[1].lower(), seqs[2][:300] + "NNNNNNNNNN" + seqs[2][310:]]
    ids += ["short", "exactk", "polyA", "lower", "withN"]
    return ids, seqs


@pytest.fixture(scope="session")
def split_index(workdir):
    """the small genomes again, written as the reference writes big genomes and big collections: genomes above --max-genome split at contig
    boundaries into chunks that are separate index entries (genomes.chunks.bin lists them), and genome batches of 5 (batch_0000 ... batch_0003)"""
    return make_index(workdir, "split", "4,4,40000,42,3", extra=("--max-genome", "30000", "--batch-size", "5"))


def read_chunk_groups(index_dir):
    import struct
    raw = open(os.path.join(index_dir, "genomes.chunks.bin"), "rb").read()
    groups, p = [], 0
    while p < len(raw):
        n = struct.unpack(">Q", raw[p:p + 8])[0]
        groups.append(list(struct.unpack(">%dQ" % n, raw[p + 8:p + 8 + 8 * n])))
        p += 8 + 8 * n
    return groups


@pytest.fixture(scope="session")
def split_queries(split_index, small_queries):
    """the small queries plus chimeras: 450 bases of one chunk followed by 450 bases of another chunk of the same split genome, so that one
    query has HSPs in two index entries that must be reported as one genome"""
    from oracle_binding import Oracle
    ids, seqs = small_queries
    o = Oracle(split_index)
    ids, seqs = list(ids), list(seqs)
    for gi, grp in enumerate(read_chunk_groups(split_index)):
        a, b = o.subseq(grp[0], 3000, 3449), o.subseq(grp[-1], 5000, 5449)
        ids.append("chimera%d" % gi)
        seqs.append(a + b)
    o.close()
    return ids, seqs


@pytest.fixture(scope="session")
def oracle_small(small_index):
    from oracle_binding import Oracle
    return Oracle(small_index)


@pytest.fixture(scope="session")
def gpu_small(small_index):
    import lexicmap_b200
    return lexicmap_b200.Index(small_index, device=0)
