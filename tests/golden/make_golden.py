#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference tools
(oracle/_ref, compiled by oracle/Makefile from /root/reference).  Run in the authoring container:

    python tests/golden/make_golden.py

Inputs are written as tests/golden/<name>.{fa,fq,fa.gz}; for each input the script stores
  <name>.com_k{3,4,5}.txt.gz        count-kmers output
  <name>.table.npz                  non-zero (keys, counts) of the 4 GiB 15mers-counts file + its sha256
  <name>.cov_bs{S}_bc{B}.txt.gz     search-15mers output for several (bin_size, bins)
The reference has no tests of its own (SURVEY.md §4); these outputs are the pins for oracle/ and
for the CUDA path.  `python tests/golden/make_golden.py --config1 [--oracle-drivers]` writes only the
digests of BASELINE.json config #1 (config1_digests).
"""
import gzip
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import oracle  # noqa: E402

COV_PARAMS = [(10, 8), (32, 10), (1, 5), (3, 1), (10, 32), (2, 3)]
CFG1 = "cfg1_100k_5kb_k3"
CFG1_SOURCES = {False: "reference tools (oracle/_ref)", True: "oracle file drivers (oracle/lrb_oracle.c)"}


def rand_seq(rng, n):
    return "".join("ACGT"[i] for i in rng.integers(0, 4, n))


def mutate(rng, s, rate):
    out = []
    for ch in s:
        u = rng.random()
        if u < rate * 0.4:
            out.append("ACGT"[rng.integers(0, 4)])
        elif u < rate * 0.7:
            out.append(ch)
            out.append("ACGT"[rng.integers(0, 4)])
        elif u < rate:
            continue
        else:
            out.append(ch)
    return "".join(out)


def revcomp_str(s):
    return s[::-1].translate(str.maketrans("ACGTacgt", "TGCAtgca"))


def build_inputs():
    files = {}
    rng = np.random.default_rng(20240611)
    base60 = rand_seq(rng, 60)
    # SURVEY.md §4 known-answer probes
    files["g01_identical25.fa"] = "".join(f">r{i}\n{base60}\n" for i in range(25))
    files["g02_identical12.fa"] = "".join(f">r{i}\n{base60}\n" for i in range(12))

    # edge cases: lengths around k, 15 and the 32-base packing blocks; N; lowercase; odd bytes
    recs = []
    recs.append(("single", rand_seq(rng, 80)))
    recs.append(("polyA20", "A" * 20))
    recs.append(("polyT33", "T" * 33))
    recs.append(("lower", rand_seq(rng, 70).lower()))
    recs.append(("mixedcase", "ACGTACGTACGTACGTACGTacgtACGTACGTACGTACGTACGTAC"))
    withn = list(rand_seq(rng, 90))
    withn[40] = "N"
    withn[41] = "N"
    withn[77] = "n"
    recs.append(("withN", "".join(withn)))
    recs.append(("empty", ""))
    for L in (1, 2, 3, 4, 5, 6, 13, 14, 15, 16, 17, 29, 30, 31, 32, 33, 34, 46, 47, 48, 63, 64, 65, 95, 96, 97, 127, 128, 129):
        recs.append((f"len{L}", rand_seq(rng, L)))
    recs.append(("allN", "N" * 50))
    recs.append(("iupac", "ACGTRYKMSWACGTACGTACGTACGTACGTBDHVACGTACGTACGTACGTACGTAC"))
    recs.append(("symbols", "ACGT-ACGT*ACGT.ACGTACGTACGTACGTACGTACGT ACGTACGTACGTACGTACGT"))
    rep = rand_seq(rng, 40)
    recs.append(("repeat", rep * 6))
    recs.append(("repeat_rc", revcomp_str(rep * 3)))
    txt = ""
    for i, (name, s) in enumerate(recs):
        if i % 3 == 0 and len(s) > 20:   # multi-line record
            txt += f">{name} some comment\n" + "\n".join(s[j:j + 17] for j in range(0, len(s), 17)) + "\n"
        else:
            txt += f">{name}\n{s}\n"
    files["g03_edge.fa"] = txt

    # FASTQ: multi-line, '@' leading a quality line, blank lines, tab in header
    fq = ""
    for i in range(12):
        s = rand_seq(rng, int(rng.integers(0, 120)))
        q = "".join(chr(33 + int(x)) for x in rng.integers(0, 41, len(s)))
        if i == 3 and len(q) > 2:
            q = "@" + q[1:]
        if i == 5:
            fq += f"@q{i}\tdesc\n" + "\n".join(s[j:j + 25] for j in range(0, len(s), 25)) + "\n+q5\n" + \
                  "\n".join(q[j:j + 31] for j in range(0, len(q), 31)) + "\n"
        else:
            fq += f"@q{i} c\n{s}\n+\n{q}\n"
        if i == 7:
            fq += "\n"
    files["g04_format.fq"] = fq

    # truncated quality: the stream stops silently at the bad record (kseq.h:214)
    s1, s2, s3 = rand_seq(rng, 50), rand_seq(rng, 60), rand_seq(rng, 70)
    files["g05_trunc.fq"] = f"@a\n{s1}\n+\n{'I' * 50}\n@b\n{s2}\n+\n{'I' * 40}\n@c\n{s3}\n+\n{'I' * 70}\n"

    # CRLF line ends, blank lines, '>' inside a line, junk before the first header, no final newline
    s = [rand_seq(rng, n) for n in (45, 100, 33, 64, 20)]
    crlf = "junk line before any header\r\n"
    crlf += f">c0 x\r\n{s[0]}\r\n"
    crlf += f">c1\r\n{s[1][:40]}\r\n\r\n{s[1][40:]}\r\n"
    crlf += f">c2\r\n{s[2][:10]}>{s[2][10:]}\r\n"
    crlf += f">c3\r\n\r\n{s[3]}\r\n"
    crlf += f">c4\r\n{s[4]}"
    files["g07_crlf.fa"] = crlf

    # '+' / '@' / '>' leading a FASTA sequence line, empty header, header-only tail
    s = [rand_seq(rng, n) for n in (50, 50, 50)]
    files["g08_leading.fa"] = f">\n{s[0]}\n>x\n{s[1][:20]}\n@{s[1][20:]}\n>y\n{s[2]}\n>tail"

    # a small community with errors, both strands, varied lengths (0..3000) -> exercises all bins
    genomes = [rand_seq(rng, n) for n in (4000, 6000, 3000)]
    weights = [30, 8, 2]
    txt = ""
    for i in range(140):
        g = int(rng.choice(3, p=np.array(weights) / sum(weights)))
        L = int(rng.choice([0, 5, 14, 15, 40, 200, 700, 1500, 3000], p=[.02, .02, .02, .02, .05, .17, .3, .3, .1]))
        st = int(rng.integers(0, len(genomes[g]) - L + 1)) if L <= len(genomes[g]) else 0
        r = genomes[g][st:st + L]
        if rng.random() < 0.5:
            r = revcomp_str(r)
        r = mutate(rng, r, 0.08)
        if rng.random() < 0.05 and len(r) > 10:
            r = r.lower()
        if rng.random() < 0.1 and len(r) > 30:
            p = int(rng.integers(0, len(r)))
            r = r[:p] + "N" + r[p + 1:]
        txt += f">read{i}\n{r}\n"
    files["g06_community.fa"] = txt
    # contigs mode (pipelines.py:139-175): 15-mers are counted on the READS (g06_community.fa) while composition and
    # coverage are computed for the FRAGMENTS of assembled contigs (runners_utils.py:53-75 split_contigs: contigs of
    # >= 5000 bases are cut into 2500-base pieces plus the last 2500 bases once more).  Written with the extension
    # .fasta so that it is not picked up as a self-contained golden input.
    contigs = [genomes[0][100:3900], genomes[1][:5600], revcomp_str(genomes[1][200:5900]), genomes[2][500:2900], genomes[0][:1200].lower()]
    frag = ""
    i = 0
    for n, c in enumerate(contigs):
        subs = [c[x:x + 2500] for x in range(0, len(c), 2500)] + [c[-2500:]] if len(c) >= 5000 else [c]
        for sc in subs:
            frag += f">{n}_{i}\n{sc}\n"
            i += 1
    files["g10_fragments.fasta"] = frag
    return files


def sha256_file(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        while True:
            b = f.read(1 << 24)
            if not b:
                break
            h.update(b)
    return h.hexdigest()


def gz_write(path, data):
    with gzip.GzipFile(path, "wb", mtime=0) as f:
        f.write(data)


def config1_digests(oracle_drivers=False):
    """BASELINE.json config #1 in full (100 k reads, 0.5 Gbases, -k 3 -bs 32 -bc 10) is too large to store: keep the size
    and sha256 of its FASTA and of the three files the tools write for it (<CFG1>.files.json).  The unmodified reference
    tools write them; only with --oracle-drivers do the oracle's file drivers, which tests/test_oracle_pins.py pins to the
    tools' files (15mers-counts by sha256 included).  `source` records which."""
    if not oracle_drivers:
        assert oracle.ref_available(), "run `make -C oracle ref` first (needs /root/reference), or pass --oracle-drivers"
    from lrbinner_b200.synth import CONFIGS, SynthSpec, write_fasta
    cfg = CONFIGS[CFG1]
    threads = os.cpu_count() or 8
    with tempfile.TemporaryDirectory(dir=os.environ.get("TMPDIR", "/tmp")) as tmp:
        fasta = os.path.join(tmp, "cfg1.fa")
        write_fasta(fasta, SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"]).host_sequences())
        com, tbl, cov = (os.path.join(tmp, x) for x in ("com_profs", "15mers-counts", "cov_profs"))
        if oracle_drivers:
            assert oracle.count_kmers_file(fasta, com, cfg["k"]) == 0
            assert oracle.count_15mers_file(fasta, tbl) == 0
            assert oracle.search_15mers_file(tbl, fasta, cov, 32, 10) == 0
        else:
            oracle.ref_count_kmers(fasta, com, cfg["k"], threads)
            oracle.ref_count_15mers(fasta, tbl, threads)
            oracle.ref_search_15mers(tbl, fasta, cov, 32, 10, threads)
        files = {name: {"bytes": os.path.getsize(p), "sha256": sha256_file(p)}
                 for name, p in (("reads.fa", fasta), ("com_profs", com), ("15mers-counts", tbl), ("cov_profs", cov))}
    source = CFG1_SOURCES[oracle_drivers]
    rec = {"workload": CFG1, "k": cfg["k"], "bin_size": 32, "bins": 10, "source": source, "files": files}
    with open(os.path.join(HERE, f"{CFG1}.files.json"), "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")
    print(f"{CFG1}: digests of the files written by the {source}", flush=True)


def main():
    if "--config1" in sys.argv:
        config1_digests(oracle_drivers="--oracle-drivers" in sys.argv)
        return
    assert oracle.ref_available(), "run `make -C oracle ref` first (needs /root/reference)"
    files = build_inputs()
    for name, txt in files.items():
        with open(os.path.join(HERE, name), "w", newline="") as f:
            f.write(txt)
    # a gzip copy of one input (gzopen path, io_utils.h:143)
    gz_write(os.path.join(HERE, "g09_community.fa.gz"), files["g06_community.fa"].encode())
    inputs = sorted([f for f in files if not f.endswith(".fasta")] + ["g09_community.fa.gz"])
    if "--contigs-only" in sys.argv:
        inputs = []
    with tempfile.TemporaryDirectory(dir=os.environ.get("TMPDIR", "/tmp")) as tmp:
        for name in inputs:
            src = os.path.join(HERE, name)
            stem = name.split(".")[0]
            for k in (3, 4, 5):
                out = os.path.join(tmp, "com")
                oracle.ref_count_kmers(src, out, k, threads=2)
                gz_write(os.path.join(HERE, f"{stem}.com_k{k}.txt.gz"), open(out, "rb").read())
            table = os.path.join(tmp, "table")
            oracle.ref_count_15mers(src, table, threads=2)
            keys, vals = oracle.table_file_sparse(table)
            np.savez_compressed(os.path.join(HERE, f"{stem}.table.npz"), keys=keys, counts=vals,
                                sha256=np.array(sha256_file(table)), file_bytes=np.array(os.path.getsize(table)))
            for bs, bc in COV_PARAMS:
                out = os.path.join(tmp, "cov")
                oracle.ref_search_15mers(table, src, out, bs, bc, threads=2)
                gz_write(os.path.join(HERE, f"{stem}.cov_bs{bs}_bc{bc}.txt.gz"), open(out, "rb").read())
            os.remove(table)
            print(f"{name}: {len(keys)} non-zero table entries", flush=True)
        # contigs mode: table of the reads, profiles of the fragments
        table = os.path.join(tmp, "table")
        frag = os.path.join(HERE, "g10_fragments.fasta")
        oracle.ref_count_15mers(os.path.join(HERE, "g06_community.fa"), table, threads=2)
        for k in (3, 4, 5):
            out = os.path.join(tmp, "com")
            oracle.ref_count_kmers(frag, out, k, threads=2)
            gz_write(os.path.join(HERE, f"g10_contigs_mode.com_k{k}.txt.gz"), open(out, "rb").read())
        for bs, bc in COV_PARAMS:
            out = os.path.join(tmp, "cov")
            oracle.ref_search_15mers(table, frag, out, bs, bc, threads=2)
            gz_write(os.path.join(HERE, f"g10_contigs_mode.cov_bs{bs}_bc{bc}.txt.gz"), open(out, "rb").read())
        os.remove(table)
        print("g10_contigs_mode: reads g06_community.fa, fragments g10_fragments.fasta", flush=True)


if __name__ == "__main__":
    main()
