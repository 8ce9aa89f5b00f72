"""tests/golden/make_golden.py -- regenerates the golden fixtures from the UNMODIFIED reference.

Run in the authoring container only (needs /root/reference and oracle/_ref built by
`make -C oracle`).  Everything it writes is committed; the GPU box never runs this.

Fixtures:
  hash_kat.json                 getHash known answers (ref_dump hash)
  wsize.json                    recommendedWindowSize for the sweep of BASELINE config 5
  stats_s{S}_k{K}.txt           minHitsRelaxed + (identity, upper bound) bit patterns per shared count
  edge_*.fa + edge_*.k{K}w{W}.mi  small hand-made sequences and the reference's minimizer records
  ecoli.k16w24.mi.sha256, ...   checksums of the full real-genome sketches
  s2e.k16.map                   all 4138 MappingResult records of Shigella -> E. coli (44 B each)
  e2s.txt / s2e.txt             fastANI_ref output lines (the reference's own goldens)
  *.fna.gz                      the two real genomes of the reference's tests/data (gzip -9)
  tricky.fq + tricky.contigs.txt  a hand-made FASTA/FASTQ mix and what the reference's kseq_read yields for it
                                (name, length, crc32 per record; `ref_dump contigs`)
  synth_ref.json                `make_golden.py synthetic` only: the seeded genome set of tests/test_oracle.py
                                (synthetic_set) through `ref_dump map` (row count + SHA-256, query fragment total per
                                query) and through fastANI_ref (output lines, FASTA directory stripped)
"""
import hashlib
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.path.join(ROOT, "oracle", "_ref")
DUMP = os.path.join(REF, "ref_dump")
CLI = os.path.join(REF, "fastANI_ref")
DATA = "/root/reference/tests/data"


def run(*a):
    return subprocess.run(list(a), capture_output=True, text=True, check=True)


def main():
    kmers = ["AAAAAAAAAAAAAAAA", "TTTTTTTTTTTTTTTT", "ACGTACGTACGTACGT", "AGCTTTTCATTCTGAC", "GTCAGAATGAAAAGCT",
             "NNNNNNNNNNNNNNNN", "ACGTNACGTACGTACG", "AGCTTTTCATTCTGACTGCAA", "ACGTA", "ACGTACGTACGTACGTACGTACGTACGTACGT",
             "ACGTACGTACGTACGTACGTACGTA", "ACGTACGTAC", "RYKMSWACGTACGTAC"]
    kat = {k: int(run(DUMP, "hash", k).stdout) for k in kmers}
    json.dump(kat, open(os.path.join(HERE, "hash_kat.json"), "w"), indent=1)

    ws = {"%d,%d" % (k, L): int(run(DUMP, "wsize", str(k), str(L)).stdout)
          for k in (16, 21) for L in (1000, 3000, 5000)}
    json.dump(ws, open(os.path.join(HERE, "wsize.json"), "w"), indent=1)

    for s, k in [(243, 16), (100, 16), (258, 16), (1, 16), (17, 21), (300, 21), (64, 16)]:
        open(os.path.join(HERE, "stats_s%d_k%d.txt" % (s, k)), "w").write(run(DUMP, "stats", str(s), str(k)).stdout)

    # ---- edge-case sequences (ragged, short, N runs, lower case, IUPAC, palindromes, repeats)
    rng = np.random.default_rng(12345)

    def rnd(n):
        return "".join("ACGT"[i] for i in rng.integers(0, 4, n))
    edge = {
        "edge_mixed": [("c0_random", rnd(5000)),
                       ("c1_short_lt_k", "ACGTACGTAC"),
                       ("c2_len_eq_w", rnd(24)),
                       ("c3_len_k_plus_w_minus_2", rnd(16 + 24 - 2)),
                       ("c4_len_k_plus_w_minus_1", rnd(16 + 24 - 1)),
                       ("c5_lower_and_N", (rnd(700).lower() + "N" * 5 + rnd(300) + "n" * 40 + rnd(800) + "NNNN" + rnd(100))),
                       ("c6_iupac", rnd(400) + "RYKMSWBDHV" + rnd(400) + "x*-" + rnd(300)),
                       ("c7_allN", "N" * 600),
                       ("c8_polyA", "A" * 900),
                       ("c9_AT_repeat", "AT" * 500),
                       ("c10_palindromes", ("ACGTACGTACGTACGT" + rnd(7)) * 40),
                       ("c11_empty_like", "A"),
                       ("c12_long_random", rnd(20000)),
                       ("c13_N_at_ends", "N" * 30 + rnd(3000) + "N" * 30),
                       ("c14_tile_edge", rnd(4050 + 16 + 24)),
                       ("c15_tile_edge2", rnd(2 * 4048 + 15))],
    }
    for name, contigs in edge.items():
        fa = os.path.join(HERE, name + ".fa")
        with open(fa, "w") as f:
            for n, s in contigs:
                f.write(">%s some description\n" % n)
                for i in range(0, len(s), 70):
                    f.write(s[i:i + 70] + "\n")
        for k, w in [(16, 24), (21, 15), (16, 13), (16, 40), (11, 5), (32, 3), (7, 1), (24, 64)]:
            out = os.path.join(HERE, "%s.k%dw%d.mi" % (name, k, w))
            run(DUMP, "sketch", str(k), str(w), out, fa)

    sums = {}
    for tag, fn in [("ecoli", "Escherichia_coli_str_K12_MG1655.fna"), ("shigella", "Shigella_flexneri_2a_01.fna")]:
        for k, w in [(16, 24), (21, 15)]:
            out = "/tmp/%s.k%dw%d.mi" % (tag, k, w)
            run(DUMP, "sketch", str(k), str(w), out, os.path.join(DATA, fn))
            b = open(out, "rb").read()
            sums["%s.k%dw%d" % (tag, k, w)] = {"records": len(b) // 12, "sha256": hashlib.sha256(b).hexdigest()}
    json.dump(sums, open(os.path.join(HERE, "sketch_sha256.json"), "w"), indent=1)

    run(DUMP, "map", "16", "3000", os.path.join(HERE, "s2e.k16.map"),
        os.path.join(DATA, "Shigella_flexneri_2a_01.fna"), os.path.join(DATA, "Escherichia_coli_str_K12_MG1655.fna"))
    msum = {}
    for k, L in [(16, 1000), (16, 5000), (21, 3000), (21, 5000)]:
        out = "/tmp/s2e.k%d.L%d.map" % (k, L)
        run(DUMP, "map", str(k), str(L), out, os.path.join(DATA, "Shigella_flexneri_2a_01.fna"),
            os.path.join(DATA, "Escherichia_coli_str_K12_MG1655.fna"))
        b = open(out, "rb").read()
        msum["s2e.k%d.L%d" % (k, L)] = {"records": len(b) // 44, "sha256": hashlib.sha256(b).hexdigest()}
    json.dump(msum, open(os.path.join(HERE, "map_sha256.json"), "w"), indent=1)

    # the reference CLI itself (its tests run from tests/ with data/ paths: fastani_tests.cpp:50-72, README.md:80)
    cwd = "/root/reference/tests"
    for tag, q, r in [("e2s", "Escherichia_coli_str_K12_MG1655.fna", "Shigella_flexneri_2a_01.fna"),
                      ("s2e", "Shigella_flexneri_2a_01.fna", "Escherichia_coli_str_K12_MG1655.fna")]:
        subprocess.run([CLI, "-q", "data/" + q, "-r", "data/" + r, "--visualize", "--matrix", "-o", "/tmp/%s.txt" % tag],
                       cwd=cwd, capture_output=True, check=True)
        for ext in ("", ".visual", ".matrix"):
            open(os.path.join(HERE, tag + ".txt" + ext), "w").write(open("/tmp/%s.txt%s" % (tag, ext)).read())
    # sweep of BASELINE config 5 on the real pair
    sweep = {}
    for k in (16, 21):
        for L in (1000, 3000, 5000):
            subprocess.run([CLI, "-q", "data/Shigella_flexneri_2a_01.fna", "-r", "data/Escherichia_coli_str_K12_MG1655.fna",
                            "-k", str(k), "--fragLen", str(L), "-o", "/tmp/sw.txt"], cwd=cwd, capture_output=True, check=True)
            sweep["%d,%d" % (k, L)] = open("/tmp/sw.txt").read().strip()
    json.dump(sweep, open(os.path.join(HERE, "sweep.json"), "w"), indent=1)
    print("golden fixtures written to", HERE)


def synthetic():
    sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
    from test_oracle import SYNTH_QUERIES, synthetic_set
    tmp = tempfile.mkdtemp()
    paths = []
    for g, contigs in enumerate(synthetic_set()):
        paths.append(os.path.join(tmp, "g%d.fa" % g))
        with open(paths[-1], "wb") as f:
            for name, seq in contigs:
                f.write(b">" + name.encode() + b" synthetic\n")
                for o in range(0, len(seq), 70):
                    f.write(seq[o:o + 70] + b"\n")
    ql, rl, out_txt, out_map = (os.path.join(tmp, n) for n in ("ql.txt", "rl.txt", "out.txt", "q.map"))
    open(ql, "w").write("\n".join(paths[i] for i in SYNTH_QUERIES) + "\n")
    open(rl, "w").write("\n".join(paths) + "\n")
    golden = {}
    for k, L in ((16, 3000), (16, 1000), (21, 5000)):
        case = {}
        for qi in SYNTH_QUERIES:
            r = run(DUMP, "map", str(k), str(L), out_map, paths[qi], *paths)
            b = open(out_map, "rb").read()
            case["q%d" % qi] = {"records": len(b) // 44, "sha256": hashlib.sha256(b).hexdigest(),
                                "total_fragments": int(re.search(r"totalQueryFragments=(\d+)", r.stderr).group(1))}
        run(CLI, "--ql", ql, "--rl", rl, "-k", str(k), "--fragLen", str(L), "-t", "2", "-o", out_txt)
        case["out_txt"] = ["\t".join(os.path.basename(f) if f.startswith(tmp) else f for f in ln.split("\t"))
                           for ln in open(out_txt).read().splitlines()]
        golden["k%d.L%d" % (k, L)] = case
    shutil.rmtree(tmp)
    json.dump(golden, open(os.path.join(HERE, "synth_ref.json"), "w"), indent=1)
    print("synth_ref.json written to", HERE)


if __name__ == "__main__":
    sys.exit(synthetic() if sys.argv[1:] == ["synthetic"] else main())
