"""CPU: the oracle (oracle/ani_oracle.c) against every golden vector produced from the UNMODIFIED
reference (tests/golden/make_golden.py) and against the reference's own test goldens."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import pyoracle as po
from conftest import GOLDEN
from fastani_b200.report import genome_length, output_lines

EC = os.path.join(GOLDEN, "Escherichia_coli_str_K12_MG1655.fna.gz")
SH = os.path.join(GOLDEN, "Shigella_flexneri_2a_01.fna.gz")


@pytest.fixture(scope="module")
def genomes():
    return po.read_fasta(EC), po.read_fasta(SH)


def test_hash_known_answers():
    kat = json.load(open(os.path.join(GOLDEN, "hash_kat.json")))
    assert len(kat) >= 12
    for kmer, want in kat.items():
        assert po.orc_hash(kmer.encode()) == want, kmer


def test_window_size_sweep():
    ws = json.load(open(os.path.join(GOLDEN, "wsize.json")))
    for key, want in ws.items():
        k, L = map(int, key.split(","))
        assert po.lib().orc_window_size(k, L) == want, key


@pytest.mark.parametrize("s,k", [(243, 16), (100, 16), (258, 16), (1, 16), (17, 21), (300, 21), (64, 16)])
def test_statistics_bit_exact(s, k):
    lines = open(os.path.join(GOLDEN, "stats_s%d_k%d.txt" % (s, k))).read().split("\n")
    assert po.lib().orc_min_hits_relaxed(s, k, 80.0) == int(lines[0])
    for x in range(s + 1):
        a, b = C.c_float(), C.c_float()
        po.lib().orc_identity(x, s, k, C.byref(a), C.byref(b))
        _, ia, ib = lines[1 + x].split()
        assert np.float32(a.value).view(np.uint32) == int(ia)
        assert np.float32(b.value).view(np.uint32) == int(ib)


@pytest.mark.parametrize("k,w", [(16, 24), (21, 15), (16, 13), (16, 40), (11, 5), (32, 3), (7, 1), (24, 64)])
def test_minimizers_edge_cases(k, w):
    """ragged / short / N-runs / lower case / IUPAC / palindromes / repeats / tile-edge lengths"""
    edge = po.read_fasta(os.path.join(GOLDEN, "edge_mixed.fa"))
    want = np.fromfile(os.path.join(GOLDEN, "edge_mixed.k%dw%d.mi" % (k, w)), dtype=po.MINIMIZER_DTYPE)
    got, by_file, _ = po.sketch_genomes([edge], k, w)
    assert len(got) == len(want) and (got == want).all()
    assert by_file.tolist() == [16]


def test_minimizers_real_genomes(genomes):
    sums = json.load(open(os.path.join(GOLDEN, "sketch_sha256.json")))
    for tag, g in zip(("ecoli", "shigella"), genomes):
        rec, _, _ = po.sketch_genomes([g], 16, 24)
        s = sums["%s.k16w24" % tag]
        assert len(rec) == s["records"]
        assert hashlib.sha256(rec.tobytes()).hexdigest() == s["sha256"]
    rec, _, _ = po.sketch_genomes([genomes[0]], 16, 24)
    assert po.Index(rec).unique() == 361568           # SURVEY section 8(c)


def test_mapping_rows_and_cgi(genomes):
    """All 4138 MappingResult records of Shigella -> E. coli, byte for byte; README.md:80 line."""
    ec, sh = genomes
    rec, sbf, lens = po.sketch_genomes([ec], 16, 24)
    rows, tot, ctr = po.map_genome(po.Index(rec), sh, 16, 24, 3000)
    want = np.fromfile(os.path.join(GOLDEN, "s2e.k16.map"), dtype=po.MAPPING_DTYPE)
    assert tot == 1608 and len(rows) == 4138
    assert rows.tobytes() == want.tobytes()
    res = po.cgi(rows, sbf, 3000)
    assert [(g, c) for g, c, _ in res] == [(0, 1303)]
    line = output_lines([(0, 0, res[0][1], tot, res[0][2])], ["data/Shigella_flexneri_2a_01.fna"],
                        ["data/Escherichia_coli_str_K12_MG1655.fna"],
                        [genome_length([len(s) for _, s in sh], 3000)], [genome_length([len(s) for _, s in ec], 3000)], 3000)
    assert line == [open(os.path.join(GOLDEN, "s2e.txt")).read().strip()]
    assert line[0].endswith("97.7507\t1303\t1608")


def test_reference_test_golden_e2s(genomes):
    """tests/fastani_tests.cpp:50-72: E. coli (query) vs Shigella (ref) = 97.664 1322 1547, and the
    .visual rows (identity, query start, ref start per 2-way mapping)."""
    ec, sh = genomes
    rec, sbf, _ = po.sketch_genomes([sh], 16, 24)
    rows, tot, _ = po.map_genome(po.Index(rec), ec, 16, 24, 3000)
    res, vis = po.cgi(rows, sbf, 3000, want_visual=True)
    assert tot == 1547 and res[0][1] == 1322
    assert "%g" % res[0][2] == "97.664"
    want = open(os.path.join(GOLDEN, "e2s.txt")).read().split("\t")
    assert want[2:] == ["97.664", "1322", "1547\n"]
    # .visual: q-start = fragment * 3000 (+0), r-start = refStartPos + offset of the ref contig
    vr, vq, vs, vi = vis
    ref_off = np.concatenate([[0], np.cumsum([len(s) for _, s in sh])])
    mine = sorted(("%g" % i, int(q) * 3000, int(s + ref_off[r])) for r, q, s, i in zip(vr, vq, vs, vi))
    gold = []
    for ln in open(os.path.join(GOLDEN, "e2s.txt.visual")):
        f = ln.rstrip("\n").split("\t")
        gold.append((f[2], int(f[6]), int(f[8])))
    gold.sort()
    # ties on identity inside one (ref contig, bin) are broken arbitrarily by std::sort in the reference:
    # identities and counts must agree everywhere, coordinates wherever the winner is unique
    assert len(mine) == len(gold) == 1322
    assert sorted(m[0] for m in mine) == sorted(g[0] for g in gold)
    assert len(set(mine) & set(gold)) >= 1300


@pytest.mark.parametrize("k,L", [(16, 1000), (16, 5000), (21, 3000), (21, 5000)])
def test_parameter_sweep(genomes, k, L):
    ec, sh = genomes
    sweep = json.load(open(os.path.join(GOLDEN, "sweep.json")))
    sums = json.load(open(os.path.join(GOLDEN, "map_sha256.json")))
    w = po.lib().orc_window_size(k, L)
    rec, sbf, _ = po.sketch_genomes([ec], k, w)
    rows, tot, _ = po.map_genome(po.Index(rec), sh, k, w, L)
    s = sums["s2e.k%d.L%d" % (k, L)]
    assert len(rows) == s["records"] and hashlib.sha256(rows.tobytes()).hexdigest() == s["sha256"]
    res = po.cgi(rows, sbf, L)
    f = sweep["%d,%d" % (k, L)].split("\t")
    assert ["%g" % res[0][2], str(res[0][1]), str(tot)] == f[2:]


def test_degenerate_k21_L1000(genomes):
    """map_stats.hpp:226-256 yields w = fragLen for k=21, fragLen=1000: no window fits, no output row."""
    ec, sh = genomes
    w = po.lib().orc_window_size(21, 1000)
    assert w == 1000
    rows, tot, _ = po.map_genome(po.Index(po.sketch_genomes([ec[:1]], 21, w)[0][:1000]), [(n, s[:50000]) for n, s in sh], 21, w, 1000)
    assert len(rows) == 0
    assert json.load(open(os.path.join(GOLDEN, "sweep.json")))["21,1000"] == ""


SYNTH_QUERIES = (0, 1, 3)


def synthetic_set():
    """Four seeded 60 kbp genomes: one multi-contig genome with lower case, an N run, a contig shorter than a fragment
    and a tandem repeat; one cut in two; two in one piece."""
    from fastani_b200.synth import synth_genome
    Lg = 60000
    genomes = []
    for g in range(4):
        a = synth_genome(21, 1 + g // 3, g % 3, 25000 * (g % 3), Lg).tobytes()
        if g == 1:
            contigs = [("g1_a", a[:21000].lower()), ("g1_tiny", a[21000:21500]), ("g1_b", a[21500:40000] + b"N" * 333 + a[40000:52000]),
                       ("g1_rep", (a[52000:52060] * 60)), ("g1_c", a[52060:])]
        elif g == 2:
            contigs = [("g2_a", a[:30011]), ("g2_b", a[30011:])]
        else:
            contigs = [("g%d" % g, a)]
        genomes.append(contigs)
    return genomes


@pytest.mark.parametrize("k,L", [(16, 3000), (16, 1000), (21, 5000)])
def test_oracle_against_the_compiled_reference_on_fresh_synthetic_genomes(k, L):
    """Beyond the real-genome fixtures: the C restatement against what the UNMODIFIED reference (oracle/_ref, compiled by
    oracle/Makefile) computed for synthetic_set() written as g0.fa ... g3.fa (tests/golden/synth_ref.json, written by
    `make_golden.py synthetic`) -- every MappingResult row byte for byte (as a SHA-256), the query fragment totals, and
    the CLI's output lines."""
    genomes = synthetic_set()
    names = ["g%d.fa" % g for g in range(len(genomes))]
    want = json.load(open(os.path.join(GOLDEN, "synth_ref.json")))["k%d.L%d" % (k, L)]
    w = po.lib().orc_window_size(k, L)
    rec, sbf, _ = po.sketch_genomes(genomes, k, w)
    ix = po.Index(rec)
    results, qlens = [], [genome_length([len(s) for _, s in g], L) for g in genomes]
    for j, qi in enumerate(SYNTH_QUERIES):
        rows, tot, _ = po.map_genome(ix, genomes[qi], k, w, L)
        ref = want["q%d" % qi]
        assert len(rows) == ref["records"] and hashlib.sha256(rows.tobytes()).hexdigest() == ref["sha256"], (qi, len(rows), ref["records"])
        assert tot == ref["total_fragments"]
        results += [(j, gid, c, tot, idn) for gid, c, idn in po.cgi(rows, sbf, L)]
    assert len(results) >= 4
    got = output_lines(results, [names[i] for i in SYNTH_QUERIES], names, [qlens[i] for i in SYNTH_QUERIES], qlens, L, 0.2)
    assert sorted(got) == sorted(want["out_txt"])
