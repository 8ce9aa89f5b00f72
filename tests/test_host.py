"""CPU: host logic of the product and the C-ABI surface (no compute calls without a GPU)."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

import fastani_b200 as fb
from conftest import GOLDEN, ROOT
from fastani_b200 import api, parallel, report
from fastani_b200.synth import synth_genome


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "fastani_b200.h")).read()
    declared = set(re.findall(r"BANI_API\s+[\w\s\*]*?\b(bani_\w+)\s*\(", hdr))
    assert len(declared) >= 28
    lib = C.CDLL(fb.library_path())
    for name in declared:
        assert hasattr(lib, name), "libfastani_b200.so does not export %s" % name
    assert declared == set(api.EXPORTED_SYMBOLS)
    fb.load_library()


def test_no_cpu_fallback():
    """The product must fail loudly without a GPU, never route through a CPU path."""
    if _has_gpu():
        pytest.skip("GPU present")
    with pytest.raises(fb.BaniError) as e:
        fb.Context(fb.Parameters())
    assert e.value.code == -2 and "no CPU fallback" in str(e.value)


def test_product_never_imports_the_oracle():
    for root, _, files in os.walk(os.path.join(ROOT, "fastani_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(root, f), errors="ignore").read()
                assert "pyoracle" not in src and "liboracle" not in src and "ani_oracle" not in src, f


def test_recommended_window_size():
    ws = json.load(open(os.path.join(GOLDEN, "wsize.json")))
    for key, want in ws.items():
        k, L = map(int, key.split(","))
        assert fb.Parameters(kmerSize=k, minReadLength=L).recommendedWindowSize() == want, key


@pytest.mark.parametrize("s,k", [(243, 16), (100, 16), (258, 16), (1, 16), (17, 21), (300, 21), (64, 16)])
def test_statistic_tables_bit_exact(s, k):
    """The (s, shared) -> identity / upper-bound table the kernels index, against the reference."""
    L = fb.load_library()
    lines = open(os.path.join(GOLDEN, "stats_s%d_k%d.txt" % (s, k))).read().split("\n")
    assert L.bani_stat_min_hits_relaxed(s, k, 80.0) == int(lines[0])
    for x in range(s + 1):
        a, b = C.c_float(), C.c_float()
        assert L.bani_stat_identity(x, s, k, C.byref(a), C.byref(b)) == 0
        _, ia, ib = lines[1 + x].split()
        assert np.float32(a.value).view(np.uint32) == int(ia)
        assert np.float32(b.value).view(np.uint32) == int(ib)


def test_argument_errors():
    L = fb.load_library()
    a, b = C.c_float(), C.c_float()
    assert L.bani_stat_identity(5, 3, 16, C.byref(a), C.byref(b)) == -1
    assert b"bad arguments" in L.bani_last_error()
    assert L.bani_ctx_sync(None) == -1


def test_fasta_reader(tmp_path):
    p = tmp_path / "x.fa"
    p.write_bytes(b">c1 desc\r\nACGT\r\nacgtn\r\n\r\n>c2\nTT TT\n@fq1\nACGTAC\n+\nIIIIII\n@fq2 x\nGG\n+\n@I\n")
    assert fb.read_fasta(str(p)) == [("c1", b"ACGTacgtn"), ("c2", b"TT TT"), ("fq1", b"ACGTAC"), ("fq2", b"GG")]     # kseq keeps inner blanks
    import gzip
    gz = tmp_path / "x.fa.gz"
    gz.write_bytes(gzip.compress(p.read_bytes()))
    assert fb.read_fasta(str(gz)) == fb.read_fasta(str(p))
    ec = fb.read_fasta(os.path.join(GOLDEN, "Escherichia_coli_str_K12_MG1655.fna.gz"))
    assert [(n, len(s)) for n, s in ec] == [("NC_000913.3", 4641652)]


def test_synth_is_deterministic_and_diverges_as_asked():
    a = synth_genome(3, 1, 0, 0, 50000)
    assert (a == synth_genome(3, 1, 0, 0, 50000)).all()
    assert set(np.unique(a)) == set(b"ACGT")
    b = synth_genome(3, 1, 5, 30000, 50000)
    assert abs(float((a != b).mean()) - 0.03) < 0.004
    assert float((a != synth_genome(3, 2, 0, 0, 50000)).mean()) > 0.7


def test_sharding_rule_matches_reference():
    # splitReferenceGenomes / correctRefGenomeIds (computeCoreIdentity.hpp:457-487)
    for n, G in [(10, 3), (2, 8), (1000, 8), (0, 2)]:
        seen = []
        for g in range(G):
            idx = parallel.shard_refs(n, G, g)
            assert idx == [j for j in range(n) if j % G == g]
            assert [parallel.global_ref_id(l, G, g) for l in range(len(idx))] == idx
            seen += idx
        assert sorted(seen) == list(range(n))


def test_output_filter_and_format():
    # sharedLength >= minGenomeLength * minFraction, float compare (computeCoreIdentity.hpp:326-332)
    rows = [(0, 0, 10, 100, np.float32(97.75071)), (0, 1, 1, 100, np.float32(99.5)), (1, 0, 20, 50, np.float32(80.0))]
    out = report.output_lines(rows, ["q0", "q1"], ["r0", "r1"], [150000, 150000], [150000, 90000], 3000, 0.2)
    assert out == ["q0\tr0\t97.7507\t10\t100", "q1\tr0\t80\t20\t50"]
    assert report.genome_length([2999, 3000, 7000], 3000) == 9000


def _cli():
    from fastani_b200 import build
    exe = os.path.join(ROOT, "fastani_b200", "bin", "fastANI")
    if not os.path.exists(exe):
        build.build_cli()
    return exe


def test_readers_have_kseq_semantics(tmp_path):
    """The C++ ingest (host/kseq_reader.hpp) and the Python reader against what the reference's own kseq_read yields
    (tests/golden/tricky.contigs.txt = `ref_dump contigs tricky.fq`): garbage before the first header, comments, CRLF,
    empty lines, FASTQ records, inner blanks, a FASTQ record whose quality spans two lines, no trailing newline."""
    import subprocess, zlib, gzip
    tricky = os.path.join(GOLDEN, "tricky.fq")
    want = [ln.split("\t") for ln in open(os.path.join(GOLDEN, "tricky.contigs.txt")).read().splitlines()]
    gz = tmp_path / "tricky.fq.gz"
    gz.write_bytes(gzip.compress(open(tricky, "rb").read()))
    for f in (tricky, str(gz)):
        r = subprocess.run([_cli(), "--dumpContigs", f], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert [ln.split("\t") for ln in r.stdout.splitlines()] == want
        assert [[n, str(len(s)), str(zlib.crc32(s) & 0xFFFFFFFF)] for n, s in fb.read_fasta(f)] == want
    for f in (os.path.join(GOLDEN, "edge_mixed.fa"), os.path.join(GOLDEN, "Shigella_flexneri_2a_01.fna.gz")):
        r = subprocess.run([_cli(), "--dumpContigs", f], capture_output=True, text=True)
        assert [ln.split("\t") for ln in r.stdout.splitlines()] == [[n, str(len(s)), str(zlib.crc32(s) & 0xFFFFFFFF)] for n, s in fb.read_fasta(f)]


def test_cli_fails_loudly_without_gpu(tmp_path):
    import subprocess
    if _has_gpu():
        pytest.skip("GPU present")
    f = os.path.join(GOLDEN, "edge_mixed.fa")
    r = subprocess.run([_cli(), "-q", f, "-r", f, "-o", str(tmp_path / "o.txt")], capture_output=True, text=True)
    assert r.returncode == 1 and "no CUDA device" in r.stderr
    r = subprocess.run([_cli(), "-q", f], capture_output=True, text=True)
    assert r.returncode == 1 and "Provide reference file" in r.stderr


def test_cli_writers_format(tmp_path):
    """cgi::outputCGI / outputPhylip of the C++ host (computeCoreIdentity.hpp:307-448) on a fixed result set: row order
    (query ascending, identity descending), float formatting (%g / %f), the minFraction filter with its float compare,
    the lower-triangular matrix with both directions averaged and self pairs ignored."""
    import subprocess
    out = tmp_path / "w.txt"
    r = subprocess.run([_cli(), "--selftestWriters", str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(out).read().splitlines() == [
        "q/a.fa\tq/a.fa\t100\t50\t50", "q/a.fa\tr/c.fa\t97.7507\t40\t50",
        "q/b.fa\tr/c.fa\t88.1235\t20\t30", "q/b.fa\tr/d.fa\t80\t6\t30",
        "r/c.fa\tr/c.fa\t100\t50\t50", "r/c.fa\tq/a.fa\t97.5\t45\t50"]
    avg = "%f" % ((np.float32(97.75071) + np.float32(97.5)) / np.float32(2))
    assert open(str(out) + ".matrix").read().splitlines() == [
        "4", "q/a.fa", "q/b.fa\tNA", "r/c.fa\t%s\t%s" % (avg, "%f" % np.float32(88.123456)), "r/d.fa\tNA\t%s\tNA" % ("%f" % np.float32(80.0))]
    # the same rows through the Python report module
    lens = {"q/a.fa": 150000, "q/b.fa": 90000, "r/c.fa": 150000, "r/d.fa": 3000000}
    q, rr = ["q/a.fa", "q/b.fa", "r/c.fa"], ["r/c.fa", "q/a.fa", "r/d.fa"]
    rows = [(0, 0, 40, 50, 97.75071), (0, 1, 50, 50, 100.0), (0, 2, 9, 50, 81.5), (1, 0, 20, 30, 88.123456), (1, 2, 6, 30, 80.0),
            (2, 1, 45, 50, 97.5), (2, 0, 50, 50, 100.0)]
    py = report.output_lines(rows, q, rr, [lens[x] for x in q], [lens[x] for x in rr], 3000, 0.2)
    assert sorted(py) == sorted(open(out).read().splitlines())


def test_bench_parity_gate_detects_every_kind_of_difference():
    """bench.py's parity gate (the rule of tests/fastani_tests.cpp:22-31) on hand-made tables: equal tables pass; a
    count, a total, an identity beyond 1e-4, a missing row and an extra row are each reported."""
    import argparse
    import bench
    names = ["c0_s0", "c0_s1", "c1_s0"]
    lens = [4998000] * 3
    cnt = np.array([[1666, 1500, 0], [1490, 1666, 0], [0, 0, 1666]], np.int32)
    idn = np.array([[100, 99.2574, 0], [99.25, 100, 0], [0, 0, 100]], np.float32)
    tot = np.array([1666, 1666, 1666], np.int64)
    ref = bench.parse_out_txt("/x/c0_s0.fna\t/x/c0_s0.fna\t100\t1666\t1666\n/x/c0_s0.fna\t/x/c0_s1.fna\t99.2574\t1500\t1666\n"
                              "/y/c1_s0.fna\t/y/c1_s0.fna\t100\t1666\t1666\n")
    ok = bench.check_parity(ref, [0, 2], [0, 1, 2], names, lens, cnt, idn, tot)
    assert ok["mismatches"] == 0 and ok["reference_rows"] == 3 and ok["pairs_checked"] == 6
    for mutate in (lambda c, i, t: c.__setitem__((0, 1), 1499), lambda c, i, t: t.__setitem__(0, 1665),
                   lambda c, i, t: i.__setitem__((0, 1), 99.2576), lambda c, i, t: c.__setitem__((0, 1), 0),
                   lambda c, i, t: c.__setitem__((2, 0), 400)):
        c2, i2, t2 = cnt.copy(), idn.copy(), tot.copy()
        mutate(c2, i2, t2)
        bad = bench.check_parity(ref, [0, 2], [0, 1, 2], names, lens, c2, i2, t2)
        assert bad["mismatches"] >= 1 and bad["example"]
    # a pair below the --minFraction output filter is not expected in the reference's file
    c2 = cnt.copy(); c2[2, 0] = 300
    assert bench.check_parity(ref, [0, 2], [0, 1, 2], names, lens, c2, idn, tot)["mismatches"] == 0
    cfg = bench.bench_config(argparse.Namespace(clusters=50, strains=20, genome_len=5000000, gpus=4))
    assert cfg["queries"] == 1000 and "4 GPU" in cfg["parallelism"]


def test_bench_output_dump(tmp_path, monkeypatch):
    """bench.py --dump-outputs: the dense tables as float arrays, exact; above the byte budget the same seeded sample of
    query rows every time, listed in query_index.npy, and the files stay within the budget."""
    import bench
    rng = np.random.default_rng(1)
    cnt = rng.integers(0, 1667, (300, 40)).astype(np.int32)
    idn = rng.uniform(80, 100, (300, 40)).astype(np.float32)
    tot = rng.integers(1, 1667, 300).astype(np.int32)
    bench.dump_outputs(str(tmp_path / "all"), cnt, idn, tot)
    ld = lambda d, n: np.load(str(tmp_path / d / (n + ".npy")))
    assert ld("all", "count_seq").dtype == np.float64 and (ld("all", "count_seq") == cnt).all()
    assert ld("all", "identity").dtype == np.float32 and (ld("all", "identity").view(np.uint32) == idn.view(np.uint32)).all()
    assert (ld("all", "total_query_fragments") == tot).all() and not (tmp_path / "all" / "query_index.npy").exists()
    monkeypatch.setattr(bench, "DUMP_BUDGET", 20000)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), cnt, idn, tot)
    q = ld("s1", "query_index").astype(np.int64)
    assert 0 < len(q) < 300 and (np.diff(q) > 0).all() and (q == ld("s2", "query_index")).all()
    assert (ld("s1", "count_seq") == cnt[q]).all() and (ld("s1", "total_query_fragments") == tot[q]).all()
    assert sum(os.path.getsize(tmp_path / "s1" / f) - 128 for f in os.listdir(tmp_path / "s1")) <= 20000     # 128 B .npy headers


def test_host_packer_matches_the_reference_bytes():
    """bani_pack_contig (no GPU): decoding the 2-bit words and patching the exception list gives back exactly the
    upper-cased bytes the reference hashes (makeUpperCase touches a-z only, commonFunc.hpp:57-66)."""
    import pyoracle as po
    rng = np.random.default_rng(12)
    seq = bytearray(rng.choice(np.frombuffer(b"ACGTacgt", np.uint8), 100003).tobytes())
    seq[5:9] = b"NNnn"; seq[40:44] = b"RYkm"; seq[16] = ord("z"); seq[31] = 0xC3; seq[32] = ord("-"); seq[100002] = ord("n")
    seq[2000:2600] = b"N" * 600
    cases = [bytes(seq), b"", b"A", b"acgtn", bytes(seq[:16]), bytes(seq[:17]), b"N" * 33,
             rng.integers(0, 256, 4099, dtype=np.uint8).tobytes(),                                  # every byte value
             bytes(rng.choice(np.frombuffer(b"ACGTacgtBDHbdhSsUu@`[{", np.uint8), 8191).tobytes())]  # neighbours of the letters in the ASCII table
    for sq in cases:
        b = fb.PackedBatch([[("x", sq)]])
        n = len(sq)
        codes = ((b.words[:(n + 15) // 16, None] >> (2 * np.arange(16, dtype=np.uint32))) & 3).reshape(-1)[:n]
        got = np.frombuffer(b"ACGT", np.uint8)[codes].copy()
        ne = int(b.exc_off[1])
        got[b.exc_pos[:ne]] = b.exc_byte[:ne]
        want = po.upper(sq)
        assert (got == want).all()
        assert ne == int(np.isin(want, np.frombuffer(b"ACGT", np.uint8), invert=True).sum())
        assert (np.diff(b.exc_pos[:ne].astype(np.int64)) > 0).all()
    # several genomes / contigs: 16-byte aligned contig starts, offsets in order; threaded packing gives the same arrays
    gl = [[("a", cases[0][:5000]), ("b", b""), ("c", cases[0][5000:9001])], [], [("d", b"acgtNNNN")]]
    b1, b2 = fb.PackedBatch(gl), fb.PackedBatch(gl, threads=3)
    assert (b1.word_off % 4 == 0).all() and list(b1.gen_off) == [0, 3, 3, 4] and list(b1.contig_len[:4]) == [5000, 0, 4001, 8]
    assert (b1.words == b2.words).all() and (b1.exc_pos == b2.exc_pos).all() and (b1.exc_off == b2.exc_off).all()


def test_records_leave_c_buffers_in_one_copy():
    """api._records_from: the structured rows of a C result buffer, bit for bit (replaces a per-field numpy copy)."""
    import ctypes as C
    from fastani_b200 import api
    rng = np.random.default_rng(5)
    for dt in (api.CGI_DTYPE, api.MAPPING_DTYPE):
        for n in (0, 1, 777):
            src = np.frombuffer(rng.integers(0, 256, n * dt.itemsize, dtype=np.uint8).tobytes(), dtype=dt)
            buf = C.create_string_buffer(src.tobytes(), max(n * dt.itemsize, 1))
            got = api._records_from(C.addressof(buf), n, dt)
            assert got.dtype == dt and got.flags.writeable and got.tobytes() == src.tobytes()


def test_identity_rows_from_dense_tables(tmp_path):
    """csrc/cgi_rows.hpp (host part of the reduction: dense count / identity tables -> cgi::CGI_Results rows, zeros skipped
    four at a time) against the plain double loop, on ragged table widths."""
    import subprocess
    src = tmp_path / "t.cpp"
    src.write_text(r'''
#include "cgi_rows.hpp"
#include <cstdio>
#include <random>
int main() {
  std::mt19937 rng(7);
  for (int nG : {0, 1, 2, 3, 4, 5, 7, 8, 9, 63, 1000}) for (int nQ : {0, 1, 3, 17}) for (int dens : {0, 1, 30, 100}) {
    std::vector<int32_t> cnt((size_t)nQ * nG); std::vector<float> idn((size_t)nQ * nG);
    for (size_t i = 0; i < cnt.size(); i++) { const bool on = (int)(rng() % 100) < dens; cnt[i] = on ? 1 + (int)(rng() % 1666) : 0; idn[i] = on ? 80.f + (rng() % 2000) / 100.f : 0.f; }
    std::vector<int32_t> qid(nQ); std::vector<uint64_t> tot(nQ);
    for (int q = 0; q < nQ; q++) { qid[q] = 1000 - q; tot[q] = 1600 + q; }
    std::vector<bani_cgi_result> got, want;
    bani::append_cgi_rows(cnt.data(), idn.data(), nQ, nG, qid.data(), tot.data(), got);
    for (int q = 0; q < nQ; q++) for (int g = 0; g < nG; g++) if (cnt[(size_t)q * nG + g] > 0) {
      bani_cgi_result r; r.refGenomeId = g; r.qryGenomeId = qid[q]; r.countSeq = cnt[(size_t)q * nG + g]; r.totalQueryFragments = (int32_t)tot[q]; r.identity = idn[(size_t)q * nG + g];
      want.push_back(r); }
    if (got.size() != want.size()) { printf("size %zu %zu nG %d nQ %d\\n", got.size(), want.size(), nG, nQ); return 1; }
    for (size_t i = 0; i < got.size(); i++) if (memcmp(&got[i], &want[i], sizeof got[i])) { printf("row %zu differs\\n", i); return 1; }
  }
  puts("ok");
  return 0;
}
''')
    exe = tmp_path / "t"
    inc = os.path.join(ROOT, "fastani_b200", "csrc")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-I", inc, str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stdout


def test_statistic_lut_rows_equal_the_scalar_functions(tmp_path):
    """StatLut (csrc/stats.cpp: rows computed by several threads, shared by the contexts of a process, binomial tails only as
    deep as they are read) against bani_stat_identity / bani_stat_min_hits_relaxed, which the goldens above pin to the reference."""
    import subprocess
    cuda_inc = "/usr/local/cuda/include"
    if not os.path.exists(os.path.join(cuda_inc, "cuda_runtime.h")):
        pytest.skip("CUDA headers not found")
    src = tmp_path / "t.cpp"
    src.write_text(r'''#include "common.cuh"
#include <cstdio>
#include <cstring>
using namespace bani;
static int check(const StatLut &l, int s, int k, float pid) {
  if (!l.have[s]) { printf("row %d missing\\n", s); return 1; }
  if (l.minHits[s] != std::max(1, stat_min_hits_relaxed(s, k, pid))) { printf("minHits %d\\n", s); return 1; }
  for (int x = 0; x <= s; x++) { float a, b; stat_identity(x, s, k, &a, &b);
    if (memcmp(&a, &l.ident[l.rowOff[s] + x], 4) || memcmp(&b, &l.upper[l.rowOff[s] + x], 4)) { printf("row %d x %d\\n", s, x); return 1; } }
  return 0;
}
int main() {
  for (int k : {16, 21}) {
    StatLut l; l.k = k; l.pid = 80.0f;
    l.ensure(97); l.ensure(130);
    for (int s = 1; s <= 130; s++) if (check(l, s, k, 80.0f)) return 1;
    if (!l.ensure_rows({700, 333, 700, 131})) return 2;
    if (l.ensure_rows({700, 333})) return 3;
    for (int s : {700, 333, 131}) if (check(l, s, k, 80.0f)) return 1;
    StatLut m; m.k = k; m.pid = 80.0f; m.ensure(130);           // second context: rows come from the process-wide cache
    if (m.ident != std::vector<float>(l.ident.begin(), l.ident.begin() + m.ident.size()) || m.minHits != std::vector<int32_t>(l.minHits.begin(), l.minHits.begin() + 131)) return 4;
  }
  puts("ok");
}
''')
    exe = tmp_path / "t"
    csrc = os.path.join(ROOT, "fastani_b200", "csrc")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-I", csrc, "-I", cuda_inc, str(src), os.path.join(csrc, "stats.cpp"), "-o", str(exe), "-lpthread"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == "ok", (r.returncode, r.stdout)


def test_upload_batches_are_assembled_in_parallel_like_in_sequence(tmp_path):
    """host/ani_host.hpp assemble_batch (the staging of host-packed genomes before bani_genome_create_packed_batch: copies made by
    several threads into uninitialised storage) against the plain back-to-back layout, genomes without contigs and empty contigs included."""
    import subprocess
    src = tmp_path / "b.cpp"
    src.write_text(r'''#include "ani_host.hpp"
#include <cstdio>
#include <random>
int main() {
  std::mt19937 rng(3);
  std::vector<bani_host::HostGenome> gs(37);
  for (auto &g : gs) {
    const int nc = rng() % 4;                                      // also genomes without contigs
    for (int c = 0; c < nc; c++) {
      bani_host::Contig ct; ct.name = "c"; ct.off = g.seq.size(); ct.len = (rng() % 5 == 0) ? 0 : rng() % 3000;
      for (uint64_t i = 0; i < ct.len; i++) g.seq.push_back("ACGTNacgtn"[rng() % ((rng() % 7 == 0) ? 10 : 4)]);
      g.contigs.push_back(ct);
    }
    skch::pack_genome(g);
  }
  std::vector<const bani_host::HostGenome *> ps; for (auto &g : gs) ps.push_back(&g);
  for (int threads : {1, 5}) for (auto range : {std::pair<size_t, size_t>{0, 37}, {3, 4}, {10, 30}}) {
    skch::HostBatch b = skch::assemble_batch(ps, range.first, range.second, threads);
    // straightforward serial statement of the same layout
    std::vector<uint32_t> w, ep; std::vector<uint8_t> eb; std::vector<int32_t> genOff(1, 0), clen; std::vector<int64_t> woff, eoff(1, 0);
    for (size_t g = range.first; g < range.second; g++) {
      const auto &G = gs[g];
      for (size_t c = 0; c < G.contigs.size(); c++) { clen.push_back((int32_t)G.contigs[c].len); woff.push_back((int64_t)w.size() + G.wordOff[c]); eoff.push_back((int64_t)ep.size() + G.excOff[c + 1]); }
      w.insert(w.end(), G.words.begin(), G.words.end()); ep.insert(ep.end(), G.excPos.begin(), G.excPos.end()); eb.insert(eb.end(), G.excByte.begin(), G.excByte.end());
      genOff.push_back((int32_t)clen.size());
    }
    clen.push_back(0); woff.push_back((int64_t)w.size());
    bool ok = b.words == w.size() && (w.empty() || !memcmp(b.w.get(), w.data(), 4 * w.size())) && genOff == b.genOff && clen == b.clen && woff == b.woff && eoff == b.eoff;
    for (int t = 0; t < 8; t++) ok = ok && b.w[b.words + t] == 0;
    ok = ok && b.ep.size() == ep.size() + 1 && std::equal(ep.begin(), ep.end(), b.ep.begin()) && std::equal(eb.begin(), eb.end(), b.eb.begin());
    if (!ok) { printf("mismatch threads %d range %zu %zu\\n", threads, range.first, range.second); return 1; }
  }
  puts("ok");
}
''')
    exe = tmp_path / "b"
    libdir = os.path.join(ROOT, "fastani_b200", "lib")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "fastani_b200", "host"), "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                        "-L", libdir, "-lfastani_b200", "-lz", "-lpthread", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == "ok", (r.returncode, r.stdout, r.stderr)
