#!/usr/bin/env python3
"""Extract small fixtures under tests/golden/ from a checkout of the reference (skani 0.3.0).  Data only: numbers
printed by the reference binary, its own sketch fixture, and small input files of its test suite.

  python tools/extract_goldens.py <skani checkout>

  g8_dist_qi_robust.tsv  <- test_results_versions/0.3.0:153-421: `skani dist -r EC590.sketch markers.bin -q o157_reads.fastq
                            --qi --robust` (tests/integration_test.rs:158-171); columns: ANI, AF_ref, AF_query, Query_name
  o157_plasmid.fasta.gz  <- test_files/o157_plasmid.fasta (gzip -9): the second contig of test_files/e.coli-o157.fasta
  o157_plasmid.sketch    <- test_files/e.coli-o157.fasta.sketch cut down to that contig: its seed positions (contig index
                            renumbered to 0), its name and length, and the markers that are canonical 21-mers ending at one of
                            its seed positions.  Seeding runs contig by contig, so this is what the reference computes for the
                            plasmid alone.
  all_ns.fa, empty_fasta.fa, list.txt, test.fasta  <- test_files/ (degenerate inputs)
  *_<n>kb.*.gz           <- the first n kb of test_files/MN-03.fa, GCF_005706655 (Bacteroides), e.coli-W, e.coli-h5 and
                            e.coli-o157 (the o157 sample also keeps the whole plasmid): inputs of G5, G6 and G7 at a size
                            that can be stored
  TOPAZ_*_60kb.fna.gz    <- contigs of the two TOPAZ eukaryotic assemblies (G9): the first IOD1 contigs up to 60 kb, and the
                            RSS1 contigs that share the most sketch k-mers with them, up to 60 kb
"""
import gzip
import os
import shutil
import struct
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
K_MARKER = 21


def g8(ref):
    lines = open(os.path.join(ref, "test_results_versions", "0.3.0")).read().split("\n")
    rows = []
    for ln in lines[151:425]:
        f = ln.split("\t")
        if len(f) == 7 and f[0].endswith("e.coli-EC590.fasta") and f[1].endswith("o157_reads.fastq"):
            rows.append((f[2], f[3], f[4], f[6]))
    assert len(rows) == 269, len(rows)
    with open(os.path.join(GOLD, "g8_dist_qi_robust.tsv"), "w") as o:
        o.write("# source: skani v0.3.0 test_results_versions/0.3.0:153-421 (dist --qi --robust, o157_reads.fastq vs EC590)\n")
        o.write("# ANI\tAF_ref\tAF_query\tQuery_name\n")
        for r in rows:
            o.write("\t".join(r) + "\n")
    print("g8_dist_qi_robust.tsv:", len(rows), "rows")


class Reader:
    def __init__(self, b):
        self.b, self.o = b, 0

    def take(self, fmt):
        v = struct.unpack_from("<" + fmt, self.b, self.o)
        self.o += struct.calcsize("<" + fmt)
        return v[0] if len(v) == 1 else v

    def string(self):
        n = self.take("Q")
        s = self.b[self.o:self.o + n]
        self.o += n
        return s


def string(s):
    return struct.pack("<Q", len(s)) + s


def canonical_marker(seq, end):
    """min(forward, reverse complement) of the 2-bit 21-mer ending at `end` (A=0 C=1 G=2 T=3; first base high)."""
    f = r = 0
    for i, ch in enumerate(seq[end - K_MARKER + 1:end + 1]):
        x = "ACGT".index(ch)
        f = (f << 2) | x
        r |= (3 - x) << (2 * i)
    return min(f, r)


def plasmid_sketch(ref):
    """Layout of the reference's legacy .sketch (bincode 1.3, little endian, u64 lengths): SURVEY.md App. C.3."""
    tf = os.path.join(ref, "test_files")
    rd = Reader(open(os.path.join(tf, "e.coli-o157.fasta.sketch"), "rb").read())
    rd.take("QQQBB")                               # c, k, marker_c, use_syncs, use_aa
    n = rd.take("Q")                               # acgt_to_aa_encoding
    rd.o += 8 * n
    n = rd.take("Q")                               # acgt_to_aa_letters
    rd.o += n
    rd.take("Q")                                   # orf_size
    head = rd.b[:rd.o]
    rd.string()                                    # file_name
    assert rd.take("B") == 1                       # Option tag
    seeds = {}
    for _ in range(rd.take("Q")):
        key = rd.take("I")
        for _ in range(rd.take("Q")):
            pos, canonical, contig, phase = rd.take("IBIB")
            if contig == 1:
                seeds.setdefault(key, []).append((pos, canonical, phase))
    contigs = [rd.string() for _ in range(rd.take("Q"))]
    rd.take("Q")                                   # total length
    lengths = [rd.take("I") for _ in range(rd.take("Q"))]
    repetitive = rd.take("Q")
    markers = set(rd.take("Q") for _ in range(rd.take("Q")))
    tail = rd.b[rd.o:]                             # trailing parameter block, kept as it is

    name, seq = open(os.path.join(tf, "o157_plasmid.fasta")).read().split("\n", 1)
    seq = seq.replace("\n", "").upper()
    assert name[1:].encode() == contigs[1] and len(seq) == lengths[1]
    ends = sorted(set(p for v in seeds.values() for p, _, _ in v))
    mine = sorted(markers & set(canonical_marker(seq, e) for e in ends))

    out = [head, string(b"o157_plasmid.fasta.gz"), b"\x01", struct.pack("<Q", len(seeds))]
    for key in sorted(seeds):
        out.append(struct.pack("<IQ", key, len(seeds[key])))
        out += [struct.pack("<IBIB", p, c, 0, ph) for p, c, ph in seeds[key]]
    out += [struct.pack("<Q", 1), string(contigs[1]), struct.pack("<QQI", lengths[1], 1, lengths[1]),
            struct.pack("<QQ", repetitive, len(mine))] + [struct.pack("<Q", m) for m in mine] + [tail]
    open(os.path.join(GOLD, "o157_plasmid.sketch"), "wb").write(b"".join(out))
    with open(os.path.join(tf, "o157_plasmid.fasta"), "rb") as i, gzip.GzipFile(
            os.path.join(GOLD, "o157_plasmid.fasta.gz"), "wb", compresslevel=9, mtime=0) as o:
        o.write(i.read())
    print("o157_plasmid.sketch: %d k-mers, %d positions, %d markers" % (len(seeds), sum(map(len, seeds.values())), len(mine)))


def degenerate(ref):
    for f in ("all_ns.fa", "empty_fasta.fa", "list.txt", "test.fasta"):
        shutil.copyfile(os.path.join(ref, "test_files", f), os.path.join(GOLD, f))


def read_fasta(path):
    op = gzip.open if path.endswith(".gz") else open
    recs = []
    for ln in op(path, "rt"):
        if ln.startswith(">"):
            recs.append([ln[1:].rstrip("\n"), []])
        else:
            recs[-1][1].append(ln.strip())
    return [(name, "".join(seq)) for name, seq in recs]


def write_fasta_gz(name, recs):
    with gzip.GzipFile(os.path.join(GOLD, name), "wb", compresslevel=9, mtime=0) as o:
        for header, seq in recs:
            o.write((">" + header + "\n" + "".join(seq[i:i + 80] + "\n" for i in range(0, len(seq), 80))).encode())
    print(name, sum(len(s) for _, s in recs), "bases")


def prefix_samples(ref):
    tf = os.path.join(ref, "test_files")
    for src, dst, kb in (("MN-03.fa", "MN-03_80kb.fa.gz", 80),
                         ("GCF_005706655.1_ASM570665v1_genomic.fna", "GCF_005706655.1_60kb.fna.gz", 60),
                         ("e.coli-W.fasta", "e.coli-W_80kb.fasta.gz", 80),
                         ("e.coli-h5.fasta", "e.coli-h5_60kb.fasta.gz", 60)):
        name, seq = read_fasta(os.path.join(tf, src))[0]
        write_fasta_gz(dst, [(name, seq[:kb * 1000])])
    (cn, cs), plasmid = read_fasta(os.path.join(tf, "e.coli-o157.fasta"))
    write_fasta_gz("e.coli-o157_60kb.fasta.gz", [(cn, cs[:60000]), plasmid])


def topaz_samples(ref, kb=60):
    import numpy as np
    import oracle_py as O
    tf = os.path.join(ref, "test_files")
    r_path, q_path = os.path.join(tf, "TOPAZ_IOD1_E001.fna.gz"), os.path.join(tf, "TOPAZ_RSS1_E007.fna.gz")
    r_recs, q_recs = read_fasta(r_path), read_fasta(q_path)
    (r,), _ = O.sketch_files([r_path])
    (q,), _ = O.sketch_files([q_path])
    er, eq = r.export(), q.export()
    r_keep, total = [], 0
    for i, (_, s) in enumerate(r_recs):
        if total >= kb * 1000:
            break
        r_keep.append(i)
        total += len(s)
    kmers = np.unique(er["kmer"][np.isin(er["cc"] >> 1, r_keep)])
    shared = np.bincount((eq["cc"] >> 1)[np.isin(eq["kmer"], kmers)], minlength=len(q_recs))
    q_keep, total = [], 0
    for i in np.argsort(-shared, kind="stable"):
        if total >= kb * 1000 or shared[i] == 0:
            break
        q_keep.append(int(i))
        total += len(q_recs[i][1])
    write_fasta_gz("TOPAZ_IOD1_E001_60kb.fna.gz", [r_recs[i] for i in r_keep])
    write_fasta_gz("TOPAZ_RSS1_E007_60kb.fna.gz", [q_recs[i] for i in sorted(q_keep)])


if __name__ == "__main__":
    ref = sys.argv[1]
    g8(ref)
    plasmid_sketch(ref)
    degenerate(ref)
    prefix_samples(ref)
    topaz_samples(ref)
