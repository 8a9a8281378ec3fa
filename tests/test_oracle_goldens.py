"""Pins the CPU oracle (oracle/) against every golden vector / known-answer test the reference holds for the
hot path (SURVEY.md section 8c, G1-G13).  Inputs come from tests/golden (data from the reference's test suite, see its
README).

G1, G5, G6, G7 and G9 are golden on whole genomes that are too large to store.  Their *_whole_genomes forms compare with the
reference's numbers and run when SKANI_TEST_FILES names the reference's test_files directory.  The tests under the
original names run the same calls on samples of those genomes stored in tests/golden (tools/extract_goldens.py).  G1's
sample is the reference's own sketch cut down to one contig.  For G5, G6, G7 and G9 the reference was not available to
run on the samples, so their expected values are the oracle's, taken when it matched the whole-genome goldens."""
import math
import os
import struct

import numpy as np
import pytest

import oracle_py as O
from conftest import needs_reference, REF_TEST_FILES as T

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def f2(x):
    """Rust `{:.2}` of an f32 product, as file_io.rs:83-96 prints it."""
    return "%.2f" % float(np.float32(x) * np.float32(100.0))


def p(name):
    return os.path.join(T, name)


def g(name):
    return os.path.join(GOLD, name)


# ---------------------------------------------------------------------------------------------------------
# G1: bit-exact seed + marker set of the o157 plasmid against the reference's own legacy .sketch fixture of
# e.coli-o157.fasta, cut down to that contig (tools/extract_goldens.py)
# ---------------------------------------------------------------------------------------------------------
def decode_legacy_sketch(path):
    """Layout: SURVEY.md App. C.3 (bincode 1.3, little endian, u64 lengths)."""
    b = open(path, "rb").read()
    o = 0

    def u64():
        nonlocal o
        v = struct.unpack_from("<Q", b, o)[0]; o += 8
        return v

    def u32():
        nonlocal o
        v = struct.unpack_from("<I", b, o)[0]; o += 4
        return v

    def u8():
        nonlocal o
        v = b[o]; o += 1
        return v

    def string():
        nonlocal o
        n = u64(); s = b[o:o + n]; o += n
        return s.decode()

    c, k, marker_c = u64(), u64(), u64()
    u8(); u8()  # use_syncs, use_aa
    n = u64(); o += 8 * n  # acgt_to_aa_encoding
    n = u64(); o += n      # acgt_to_aa_letters
    u64()                  # orf_size
    file_name = string()
    assert u8() == 1       # Option tag
    nk = u64()
    recs = []
    for _ in range(nk):
        key = u32()
        ln = u64()
        for _ in range(ln):
            pos = u32(); canonical = u8(); contig = u32(); u8()  # phase
            recs.append((key, pos, contig, canonical))
    ncont = u64(); contigs = [string() for _ in range(ncont)]
    total = u64()
    ncl = u64(); cl = [u32() for _ in range(ncl)]
    u64()  # repetitive_kmers
    nm = u64(); markers = [u64() for _ in range(nm)]
    return dict(c=c, k=k, marker_c=marker_c, file_name=file_name, nk=nk, recs=recs, contigs=contigs, total=total,
                contig_lengths=cl, markers=markers)


def check_seed_fixture(sketch, fasta, n_kmers, n_records, n_markers, contig_lengths):
    ref = decode_legacy_sketch(sketch)
    assert (ref["c"], ref["k"], ref["marker_c"]) == (125, 15, 1000)
    sk, _ = O.sketch_files([fasta])
    s = sk[0]
    assert s.n_kmers == ref["nk"] == n_kmers
    assert s.n_records == len(ref["recs"]) == n_records
    assert s.n_markers == len(ref["markers"]) == n_markers
    e = s.export()
    assert list(e["contig_lengths"]) == ref["contig_lengths"] == contig_lengths
    ours = sorted(zip(e["kmer"].tolist(), e["pos"].tolist(), (e["cc"] >> 1).tolist(), (e["cc"] & 1).tolist()))
    assert ours == sorted(ref["recs"])
    assert e["markers"].tolist() == sorted(ref["markers"])
    assert s.total_len == ref["total"]
    assert [s.contig_name(i) for i in range(len(contig_lengths))] == ref["contigs"]


def test_g1_seed_fixture_bit_exact():
    check_seed_fixture(g("o157_plasmid.sketch"), g("o157_plasmid.fasta.gz"), 730, 759, 81, [92596])


@needs_reference
def test_g1_seed_fixture_bit_exact_whole_genome():
    check_seed_fixture(p("e.coli-o157.fasta.sketch"), p("e.coli-o157.fasta"), 40716, 44127, 5073, [5416633, 92596])


# G2: tests/tests.rs:130-144 -- AVX2 path == scalar path on the 120-base string, c = 10
def test_g2_avx2_equals_scalar():
    s = b"ATCAGATTTAAAAAAAAATTTTGCTAGCTGATCGATCGATCGATGTGTATATATTAAAAGAGAGAGAGGGGGGGGAAAAAAAAAAAAACTGATCGATCGATGCTAGCTAGTCAGTCGATG"
    assert len(s) == 120
    L = O.lib()
    buf = np.frombuffer(s, np.uint8)
    # the seeders are called directly (no MIN_LENGTH_CONTIG rule), as tests/tests.rs does
    a = O.Sketch(L.orc_seed_one_contig(buf.ctypes.data, len(s), 10, 15, 1000, 1))
    b = O.Sketch(L.orc_seed_one_contig(buf.ctypes.data, len(s), 10, 15, 1000, 0))
    ea, eb = a.export(), b.export()
    assert a.n_records > 0
    for key in ("kmer", "pos", "cc", "markers"):
        assert np.array_equal(ea[key], eb[key])


# G3: tests/tests.rs:149-157 -- 154 x 'N' + 'n', c = 30, scalar path -> zero seeds
def test_g3_all_n_scalar():
    s = b"N" * 154 + b"n"
    buf = np.frombuffer(s, np.uint8)
    a = O.Sketch(O.lib().orc_seed_one_contig(buf.ctypes.data, len(s), 30, 15, 1000, 0))
    assert a.n_kmers == 0


def test_g4_dist_fast_ec590_k12():
    # test_results_versions/0.3.0:121  (`dist EC590 K12 --fast -n 3`; first positional is the query)
    r, _ = O.sketch_files([g("e.coli-K12.fasta.gz")], c=200)
    q, _ = O.sketch_files([g("e.coli-EC590.fasta.gz")], c=200)
    res = O.dist(r, q, O.cmd(learned_ani=True))
    assert len(res) == 1
    assert (f2(res[0].ani), f2(res[0].af_ref), f2(res[0].af_query)) == ("99.42", "94.47", "95.06")


def test_g5_dist_c30_k12_klebsiella():
    r, _ = O.sketch_files([g("MN-03_80kb.fa.gz")], c=30)
    q, _ = O.sketch_files([g("e.coli-K12.fasta.gz")], c=30)
    res = O.dist(r, q, O.cmd(learned_ani=False))
    assert [(f2(x.ani), f2(x.af_ref), f2(x.af_query)) for x in res] == [("81.23", "23.73", "0.41")]


@needs_reference
def test_g5_dist_c30_k12_klebsiella_whole_genomes():
    # test_results_versions/0.3.0:125 (`dist K12 MN-03 -c 30`: learned ANI off because c < 70)
    r, _ = O.sketch_files([p("MN-03.fa")], c=30)
    q, _ = O.sketch_files([p("e.coli-K12.fasta")], c=30)
    res = O.dist(r, q, O.cmd(learned_ani=False))
    assert (f2(res[0].ani), f2(res[0].af_ref), f2(res[0].af_query)) == ("79.68", "26.21", "29.59")


def test_g6_triangle_query_list():
    files = [g("o157_reads.fa.gz"), g("e.coli-EC590.fasta.gz"), g("e.coli-W_80kb.fasta.gz"), g("GCF_005706655.1_60kb.fna.gz")]
    sk, _ = O.sketch_files(files)
    names = [os.path.basename(s.file_name) for s in sk]
    assert names == ["GCF_005706655.1_60kb.fna.gz", "e.coli-EC590.fasta.gz", "e.coli-W_80kb.fasta.gz", "o157_reads.fa.gz"]
    res, info = O.triangle(sk, O.cmd(learned_ani=True))
    got = {(r.ref_id, r.query_id): f2(r.ani) for r in res}
    assert got == {(1, 2): "98.40", (1, 3): "92.81", (2, 3): "92.15"}
    assert info["n_chained"] == 3  # the Bacteroides sample fails the marker screen against all three


@needs_reference
def test_g6_triangle_query_list_whole_genomes():
    # test_results_versions/0.3.0:98-102: sorted file order GCF_005706655, EC590, W.gz, reads.fastq
    files = [p("o157_reads.fastq"), p("e.coli-EC590.fasta"), p("e.coli-W.fasta.gz"),
             p("GCF_005706655.1_ASM570665v1_genomic.fna")]
    sk, _ = O.sketch_files(files)
    names = [os.path.basename(s.file_name) for s in sk]
    assert names == ["GCF_005706655.1_ASM570665v1_genomic.fna", "e.coli-EC590.fasta", "e.coli-W.fasta.gz", "o157_reads.fastq"]
    res, info = O.triangle(sk, O.cmd(learned_ani=True))
    got = {(r.ref_id, r.query_id): f2(r.ani) for r in res}
    assert got == {(1, 2): "98.58", (1, 3): "92.81", (2, 3): "93.15"}
    assert info["n_chained"] == 3  # GCF_005706655 fails the marker screen against all three


def test_g7_search_median():
    refs_files = ["e.coli-EC590.fasta.gz", "e.coli-h5_60kb.fasta.gz", "e.coli-K12.fasta.gz", "e.coli-o157_60kb.fasta.gz",
                  "e.coli-W_80kb.fasta.gz", "o157_plasmid.fasta.gz", "o157_reads.fa.gz", "test.fasta"]
    refs, nwarn = O.sketch_files([g(f) for f in refs_files])
    assert len(refs) == 7 and nwarn == 1  # test.fasta is below the minimum length
    q, _ = O.sketch_files([g("e.coli-o157_60kb.fasta.gz")])
    res = O.search(refs, q, O.cmd(median=True, learned_ani=False, min_af=-1.0, rescue_small=False))
    rows = {os.path.basename(refs[r.ref_id].file_name): (f2(r.ani), f2(r.af_ref), f2(r.af_query)) for r in res}
    assert rows == {"e.coli-o157_60kb.fasta.gz": ("100.00", "99.72", "99.72"),
                    "o157_plasmid.fasta.gz": ("100.00", "99.84", "60.58"),
                    "e.coli-EC590.fasta.gz": ("96.70", "0.91", "27.59"),
                    "e.coli-K12.fasta.gz": ("96.64", "0.86", "26.10"),
                    "o157_reads.fa.gz": ("92.75", "1.34", "48.52")}


@needs_reference
def test_g7_search_median_whole_genomes():
    # test_results_versions/0.3.0:131-135 (`search --median -n 5`, o157 vs DB of list.txt; no marker index)
    refs_files = ["e.coli-EC590.fasta", "e.coli-h5.fasta", "e.coli-K12.fasta", "e.coli-o157.fasta", "e.coli-W.fasta",
                  "e.coli-W.fasta.gz", "o157_plasmid.fasta", "o157_reads.fastq", "test.fasta"]
    refs, nwarn = O.sketch_files([p(f) for f in refs_files])
    q, _ = O.sketch_files([p("e.coli-o157.fasta")])
    res = O.search(refs, q, O.cmd(median=True, learned_ani=False, min_af=-1.0, rescue_small=False))
    rows = {os.path.basename(refs[r.ref_id].file_name): (f2(r.ani), f2(r.af_ref), f2(r.af_query)) for r in res}
    top = sorted(rows.items(), key=lambda kv: -float(kv[1][0]))
    assert rows["o157_plasmid.fasta"] == ("100.00", "99.84", "1.68")
    assert rows["e.coli-o157.fasta"] == ("100.00", "100.00", "100.00")
    assert rows["e.coli-EC590.fasta"] == ("98.44", "87.84", "73.62")
    assert rows["e.coli-K12.fasta"] == ("98.42", "88.04", "74.25")
    assert rows["e.coli-W.fasta"] == ("98.39", "85.46", "75.97")


def test_g8_dist_qi_robust_269_rows():
    gold = {}
    for ln in open(os.path.join(GOLD, "g8_dist_qi_robust.tsv")):
        if ln.startswith("#"):
            continue
        ani, afr, afq, name = ln.rstrip("\n").split("\t")
        gold[name] = (ani, afr, afq)
    assert len(gold) == 269
    refs, _ = O.sketch_files([g("e.coli-EC590.fasta.gz")])
    # o157_reads.fastq with the quality lines dropped (same ids, same sequences)
    qs, _ = O.sketch_files([g("o157_reads.fa.gz")], individual=True)
    assert len(qs) == 364
    # --qi: marker index on (parse.rs:750), learned ANI off (regression.rs:8-10), --robust
    res = O.dist(refs, qs, O.cmd(robust=True, learned_ani=False), use_index=True)
    got = {qs[r.query_id].contig_name(0): (f2(r.ani), f2(r.af_ref), f2(r.af_query)) for r in res}
    assert len(got) == 269
    assert got == gold


def f32s(x):  # Rust {:?} of f32 = shortest round-trip repr
    return np.format_float_positional(np.float32(x), unique=True, trim="-")


def test_g9_eukaryote_full_struct():
    r, _ = O.sketch_files([g("TOPAZ_IOD1_E001_60kb.fna.gz")])
    q, _ = O.sketch_files([g("TOPAZ_RSS1_E007_60kb.fna.gz")])
    res = O.chain(r[0], q[0], O.cmd(learned_ani=True))
    assert [f32s(getattr(res, f)) for f in ("ani", "af_query", "af_ref", "ci_upper", "ci_lower", "std")] == \
        ["0.99336547", "0.72314334", "0.7482639", "0.9955625", "0.9908015", "0.005323155"]
    assert (res.q90_q, res.q90_r, res.q50_q, res.q50_r, res.q10_q, res.q10_r) == (7526.0, 7780.0, 4957.0, 3730.0, 3310.0, 2699.0)
    assert (res.num_contigs_q, res.num_contigs_r, res.avg_chain_int_len, res.total_bases_covered) == (12, 14, 3798, 45579)
    raw = O.chain(r[0], q[0], O.cmd(learned_ani=False))
    assert raw.ani >= 0.98 and res.ani <= raw.ani  # tests/tests.rs:112-126


@needs_reference
def test_g9_eukaryote_full_struct_whole_genomes():
    # test_results_versions/0.3.0:448, tests/tests.rs:82-128
    r, _ = O.sketch_files([p("TOPAZ_IOD1_E001.fna.gz")])
    q, _ = O.sketch_files([p("TOPAZ_RSS1_E007.fna.gz")])
    res = O.chain(r[0], q[0], O.cmd(learned_ani=True))
    assert f32s(res.ani) == "0.9898663"
    assert f32s(res.af_query) == "0.60535073"
    assert f32s(res.af_ref) == "0.74593395"
    assert f32s(res.ci_upper) == "0.9900135"
    assert f32s(res.ci_lower) == "0.9897283"
    assert f32s(res.std) == "0.007433527"
    assert (res.q90_q, res.q90_r, res.q50_q, res.q50_r, res.q10_q, res.q10_r) == (9095.0, 7016.0, 4276.0, 3761.0, 2759.0, 2688.0)
    assert (res.num_contigs_q, res.num_contigs_r, res.avg_chain_int_len, res.total_bases_covered) == (8559, 8377, 3187, 27655368)
    raw = O.chain(r[0], q[0], O.cmd(learned_ani=False))
    assert raw.ani >= 0.98 and res.ani <= raw.ani  # tests/tests.rs:112-126


def test_g10_result_counts_on_reads():
    # test_results_versions/0.3.0:60-69, tests/int_test_new.rs:56-133
    reads = [g("o157_reads.fa.gz")]
    ind, _ = O.sketch_files(reads, individual=True)
    res, _ = O.triangle(ind, O.cmd(learned_ani=False, rescue_small=True))          # triangle -i -E
    assert len(res) == 270
    res, _ = O.triangle(ind, O.cmd(learned_ani=False, rescue_small=False))         # --faster-small
    assert len(res) == 154
    big, _ = O.sketch_files(reads, individual=True, marker_c=1000000)
    res, _ = O.triangle(big, O.cmd(learned_ani=False, screen_val=0.95))            # -s 95 -m 1000000
    assert len(res) == 345
    big2, _ = O.sketch_files(reads, individual=True, marker_c=10000000)
    res, _ = O.triangle(big2, O.cmd(learned_ani=False))                            # -m 10000000
    assert len(res) == 345
    ref, _ = O.sketch_files([g("e.coli-EC590.fasta.gz")])
    # dist --qi: index on
    assert len(O.dist(ref, ind, O.cmd(learned_ani=False, rescue_small=False), use_index=True)) == 175
    assert len(O.dist(ref, ind, O.cmd(learned_ani=False, rescue_small=True), use_index=True)) == 269
    assert len(O.dist(ref, ind, O.cmd(learned_ani=False, rescue_small=False, screen_val=0.95), use_index=True)) == 87
    refb, _ = O.sketch_files([g("e.coli-EC590.fasta.gz")], marker_c=10000000000)
    indb, _ = O.sketch_files(reads, individual=True, marker_c=10000000000)
    assert len(O.dist(refb, indb, O.cmd(learned_ani=False, rescue_small=False), use_index=True)) == 0


def test_g11_self_vs_self():
    # tests/tests.rs:57-59 holds for any genome; it is checked on K12 here (the reference uses e.coli-W, not stored)
    r, _ = O.sketch_files([g("e.coli-K12.fasta.gz")])
    res = O.chain(r[0], r[0], O.cmd(learned_ani=False))
    assert res.ani >= 1.0 and res.af_query >= 0.99 and res.af_ref >= 0.99


def test_g12_viruses_small_genomes():
    # tests/int_test_new.rs:58-81: row0 in (99.0, 99.9), row1 > 99.9, with and without --faster-small;
    # --small-genomes == -c 30 -m 200 --faster-small (parse.rs:847-853)
    for kw, cp in [(dict(), O.cmd(learned_ani=False)), (dict(), O.cmd(learned_ani=False, rescue_small=False)),
                   (dict(c=30, marker_c=200), O.cmd(learned_ani=False, rescue_small=False))]:
        sk, _ = O.sketch_files([g("viruses.fna")], individual=True, **kw)
        assert len(sk) == 3
        res, _ = O.triangle(sk, cp)
        got = {(r.ref_id, r.query_id): r.ani * 100 for r in res}
        assert set(got) == {(0, 1), (0, 2), (1, 2)}
        assert 99.0 < got[(0, 1)] < 99.9
        assert got[(0, 2)] > 99.9 and got[(1, 2)] > 99.9


def test_g13_readme_example_config1():
    # README.md:48,142 / BASELINE.json configs[0]: `skani dist refs/e.coli-EC590.fasta refs/e.coli-K12.fasta`
    r, _ = O.sketch_files([g("e.coli-K12.fasta.gz")])
    q, _ = O.sketch_files([g("e.coli-EC590.fasta.gz")])
    res = O.dist(r, q, O.cmd(learned_ani=True))
    assert (f2(res[0].ani), f2(res[0].af_ref), f2(res[0].af_query)) == ("99.39", "91.89", "92.46")


def test_degenerate_inputs():
    # tests/int_test_new.rs:135-163: missing file, non-FASTA, all < 500 bp, all-N produce no sketches / no rows
    sk, nwarn = O.sketch_files([g("does_not_exist.fa"), g("list.txt"), g("test.fasta"), g("empty_fasta.fa")])
    assert len(sk) == 0 and nwarn == 4
    sk, _ = O.sketch_files([g("all_ns.fa")])
    assert len(sk) == 1 and sk[0].n_records == 0 and sk[0].n_markers == 0
    res, _ = O.triangle(sk + sk, O.cmd())
    assert len(res) == 0
