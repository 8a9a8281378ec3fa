"""ctypes binding of the CPU oracle (oracle/liboracle.so).  TEST INFRASTRUCTURE ONLY."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB_PATH = os.path.join(ORACLE_DIR, "liboracle.so")


class OrcResult(C.Structure):
    _fields_ = [(n, C.c_float) for n in
                ("ani", "af_query", "af_ref", "ci_lower", "ci_upper", "std",
                 "q90_q", "q90_r", "q50_q", "q50_r", "q10_q", "q10_r")] + \
               [(n, C.c_uint32) for n in
                ("num_contigs_q", "num_contigs_r", "avg_chain_int_len", "total_bases_covered", "ref_id", "query_id")]


class OrcCmd(C.Structure):
    _fields_ = [("screen_val", C.c_double), ("min_aligned_frac", C.c_double), ("both_min_aligned_frac", C.c_double),
                ("robust", C.c_int32), ("median", C.c_int32), ("learned_ani", C.c_int32), ("rescue_small", C.c_int32)]


def cmd(screen_val=0.0, min_af=0.15, both_min_af=-0.01, robust=False, median=False, learned_ani=True,
        rescue_small=True):
    return OrcCmd(screen_val, min_af, both_min_af, int(robust), int(median), int(learned_ani), int(rescue_small))


_lib = None


def build():
    subprocess.check_call(["make", "-s", "-C", ORACLE_DIR])


def build_native():
    """-march=native build for the CPU baseline, made in a new temporary directory (the tree may be read-only) that is
    removed at exit; returns the library's path or None."""
    try:
        d = tempfile.mkdtemp(prefix="skani-oracle-native-")
        atexit.register(shutil.rmtree, d, True)
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "native", "NATIVE_DIR=" + d])
        return os.path.join(d, "liboracle.so")
    except Exception:
        return None


def use_library(path):
    """Bind a specific build of the oracle (bench.py --impl reference: the -march=native one). Call before lib()."""
    global LIB_PATH, _lib
    LIB_PATH, _lib = path, None


def set_avx2_intrinsics(on=True):
    """Seeding with the reference's 4-lane AVX2 instruction mix (baseline timing); returns whether it is active."""
    return bool(lib().orc_set_avx2_intrinsics(int(on)))


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        build()
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i32, dbl = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_double
    L.orc_mm_hash64.restype = u64; L.orc_mm_hash64.argtypes = [u64]
    L.orc_set_avx2_intrinsics.restype = i32; L.orc_set_avx2_intrinsics.argtypes = [i32]
    L.orc_sketch_files.restype = i32
    L.orc_sketch_files.argtypes = [C.POINTER(C.c_char_p), i32, u64, u64, u64, i32, i32, i32,
                                   C.POINTER(C.POINTER(vp)), C.POINTER(i32), C.POINTER(i32)]
    L.orc_free_array.argtypes = [vp]
    L.orc_sketch_from_contigs.restype = vp
    L.orc_sketch_from_contigs.argtypes = [C.c_char_p, vp, vp, u32, u64, u64, u64, i32]
    L.orc_sketch_free.argtypes = [vp]
    L.orc_sketch_many.restype = i32
    L.orc_sketch_many.argtypes = [vp, vp, vp, u32, u32, u64, u64, u64, i32, C.POINTER(vp)]
    L.orc_seed_one_contig.restype = vp
    L.orc_seed_one_contig.argtypes = [vp, u64, u64, u64, u64, i32]
    L.orc_time_seeding.restype = dbl
    L.orc_time_seeding.argtypes = [vp, vp, u32, u64, u64, u64, i32]
    for f in ("n_records", "n_kmers", "n_markers", "n_contigs", "total_len", "contig_order"):
        fn = getattr(L, "orc_sketch_" + f); fn.restype = u64; fn.argtypes = [vp]
    L.orc_sketch_file_name.restype = C.c_char_p; L.orc_sketch_file_name.argtypes = [vp]
    L.orc_sketch_contig_name.restype = C.c_char_p; L.orc_sketch_contig_name.argtypes = [vp, u64]
    L.orc_sketch_export.argtypes = [vp] * 6
    L.orc_check_markers_quickly.restype = i32; L.orc_check_markers_quickly.argtypes = [vp, vp, dbl, i32]
    L.orc_screen_triangle.restype = i32
    L.orc_screen_triangle.argtypes = [C.POINTER(vp), i32, dbl, i32, C.POINTER(C.POINTER(u64)), C.POINTER(C.POINTER(u32))]
    L.orc_chain.restype = i32; L.orc_chain.argtypes = [vp, vp, C.POINTER(OrcCmd), C.POINTER(OrcResult)]
    L.orc_chain_debug.restype = vp; L.orc_chain_debug.argtypes = [vp, vp, C.POINTER(OrcCmd)]
    L.orc_debug_free.argtypes = [vp]
    L.orc_debug_result.argtypes = [vp, C.POINTER(OrcResult)]
    L.orc_debug_switched.restype = i32; L.orc_debug_switched.argtypes = [vp]
    for f in ("n_anchors", "n_chunks", "n_intervals", "n_ests"):
        fn = getattr(L, "orc_debug_" + f); fn.restype = u64; fn.argtypes = [vp]
    L.orc_debug_anchors.argtypes = [vp] * 4
    L.orc_debug_chunks.argtypes = [vp] * 3
    L.orc_debug_intervals.argtypes = [vp] * 2
    L.orc_debug_ests.argtypes = [vp] * 3
    L.orc_gbdt_predict.restype = C.c_float; L.orc_gbdt_predict.argtypes = [i32, vp]
    L.orc_triangle.restype = i32
    L.orc_triangle.argtypes = [C.POINTER(vp), i32, C.POINTER(OrcCmd), i32, C.POINTER(C.POINTER(OrcResult)),
                               C.POINTER(u64), C.POINTER(u64), C.POINTER(dbl), C.POINTER(dbl)]
    for f in ("orc_dist", "orc_search"):
        fn = getattr(L, f); fn.restype = i32
        fn.argtypes = [C.POINTER(vp), i32, C.POINTER(vp), i32, C.POINTER(OrcCmd), i32, i32,
                       C.POINTER(C.POINTER(OrcResult)), C.POINTER(u64)]
    _lib = L
    return L


class Sketch:
    def __init__(self, handle):
        self.h = C.c_void_p(handle)

    def __del__(self):
        try:
            lib().orc_sketch_free(self.h)
        except Exception:
            pass

    @property
    def file_name(self): return lib().orc_sketch_file_name(self.h).decode()
    def contig_name(self, i=0): return lib().orc_sketch_contig_name(self.h, i).decode()
    @property
    def n_records(self): return lib().orc_sketch_n_records(self.h)
    @property
    def n_kmers(self): return lib().orc_sketch_n_kmers(self.h)
    @property
    def n_markers(self): return lib().orc_sketch_n_markers(self.h)
    @property
    def n_contigs(self): return lib().orc_sketch_n_contigs(self.h)
    @property
    def total_len(self): return lib().orc_sketch_total_len(self.h)

    def export(self):
        n, m, nc = self.n_records, self.n_markers, self.n_contigs
        kmer = np.zeros(n, np.uint32); pos = np.zeros(n, np.uint32); cc = np.zeros(n, np.uint32)
        mk = np.zeros(m, np.uint64); cl = np.zeros(nc, np.uint32)
        lib().orc_sketch_export(self.h, kmer.ctypes.data, pos.ctypes.data, cc.ctypes.data, mk.ctypes.data, cl.ctypes.data)
        return dict(kmer=kmer, pos=pos, cc=cc, markers=mk, contig_lengths=cl)


def sketch_files(paths, c=125, k=15, marker_c=1000, individual=False, avx2sem=True, threads=4):
    L = lib()
    arr = (C.c_char_p * len(paths))(*[p.encode() for p in paths])
    out = C.POINTER(C.c_void_p)(); n = C.c_int(); nw = C.c_int()
    rc = L.orc_sketch_files(arr, len(paths), c, k, marker_c, int(individual), int(avx2sem), threads,
                            C.byref(out), C.byref(n), C.byref(nw))
    if rc != 0:
        raise ValueError("orc_sketch_files rc=%d" % rc)
    sk = [Sketch(out[i]) for i in range(n.value)]
    L.orc_free_array(out)
    return sk, nw.value


def sketch_from_contigs(name, seqs, c=125, k=15, marker_c=1000, avx2sem=True):
    """seqs: list of bytes/np.uint8 arrays (ASCII)."""
    arrs = [np.frombuffer(s, np.uint8) if isinstance(s, (bytes, bytearray)) else np.asarray(s, np.uint8) for s in seqs]
    off = np.zeros(len(arrs) + 1, np.uint64)
    off[1:] = np.cumsum([len(a) for a in arrs])
    buf = np.concatenate(arrs) if arrs else np.zeros(0, np.uint8)
    buf = np.ascontiguousarray(buf)
    h = lib().orc_sketch_from_contigs(name.encode(), buf.ctypes.data, off.ctypes.data, len(arrs), c, k, marker_c, int(avx2sem))
    return Sketch(h)


def sketch_many(bases, contig_off, genome_of_contig, n_genomes, c=125, k=15, marker_c=1000, threads=4):
    """Oracle sketches of genomes laid out like sk_sketch_batch's input; OpenMP threads over genomes."""
    bases = np.ascontiguousarray(bases, np.uint8)
    off = np.ascontiguousarray(contig_off, np.uint64); goc = np.ascontiguousarray(genome_of_contig, np.uint32)
    out = (C.c_void_p * n_genomes)()
    lib().orc_sketch_many(bases.ctypes.data, off.ctypes.data, goc.ctypes.data, len(goc), n_genomes, c, k, marker_c, threads, out)
    return [Sketch(out[i]) for i in range(n_genomes)]


def chain(ref, query, cp=None):
    cp = cp or cmd()
    r = OrcResult()
    lib().orc_chain(ref.h, query.h, C.byref(cp), C.byref(r))
    return r


def chain_debug(ref, query, cp=None):
    cp = cp or cmd()
    L = lib()
    d = C.c_void_p(L.orc_chain_debug(ref.h, query.h, C.byref(cp)))
    try:
        res = OrcResult(); L.orc_debug_result(d, C.byref(res))
        na, nc, ni, ne = (L.orc_debug_n_anchors(d), L.orc_debug_n_chunks(d), L.orc_debug_n_intervals(d), L.orc_debug_n_ests(d))
        a5 = np.zeros((na, 5), np.uint32); score = np.zeros(na, np.int64); ptr = np.zeros(na, np.uint32)
        L.orc_debug_anchors(d, a5.ctypes.data, score.ctypes.data, ptr.ctypes.data)
        first = np.zeros(nc + 1, np.uint32); nseeds = np.zeros(nc, np.uint32)
        if nc:
            L.orc_debug_chunks(d, first.ctypes.data, nseeds.ctypes.data)
        iv = np.zeros((ni, 11), np.int64)
        L.orc_debug_intervals(d, iv.ctypes.data)
        est = np.zeros(ne, np.float64); w = np.zeros(ne, np.uint64)
        L.orc_debug_ests(d, est.ctypes.data, w.ctypes.data)
        return dict(result=res, switched=bool(L.orc_debug_switched(d)), anchors=a5, score=score, pointer=ptr,
                    chunk_first=first, chunk_nseeds=nseeds, intervals=iv, est=est, weight=w)
    finally:
        L.orc_debug_free(d)


def _results(out, n):
    res = [OrcResult.from_buffer_copy(out[i]) for i in range(n.value)]
    lib().orc_free_array(out)
    return res


def triangle(sketches, cp=None, threads=4):
    cp = cp or cmd()
    L = lib()
    hs = (C.c_void_p * len(sketches))(*[s.h for s in sketches])
    out = C.POINTER(OrcResult)(); n = C.c_uint64(); nch = C.c_uint64(); ts = C.c_double(); tc = C.c_double()
    L.orc_triangle(hs, len(sketches), C.byref(cp), threads, C.byref(out), C.byref(n), C.byref(nch), C.byref(ts), C.byref(tc))
    return _results(out, n), dict(n_chained=nch.value, t_screen=ts.value, t_chain=tc.value)


def _qr(fn, refs, queries, cp, use_index, threads):
    cp = cp or cmd()
    hr = (C.c_void_p * len(refs))(*[s.h for s in refs])
    hq = (C.c_void_p * len(queries))(*[s.h for s in queries])
    out = C.POINTER(OrcResult)(); n = C.c_uint64()
    fn(hr, len(refs), hq, len(queries), C.byref(cp), int(use_index), threads, C.byref(out), C.byref(n))
    return _results(out, n)


def dist(refs, queries, cp=None, use_index=False, threads=4):
    return _qr(lib().orc_dist, refs, queries, cp, use_index, threads)


def search(refs, queries, cp=None, use_index=False, threads=4):
    return _qr(lib().orc_search, refs, queries, cp, use_index, threads)


def screen_triangle(sketches, screen_val=0.0, rescue_small=True):
    L = lib()
    hs = (C.c_void_p * len(sketches))(*[s.h for s in sketches])
    ro = C.POINTER(C.c_uint64)(); cols = C.POINTER(C.c_uint32)()
    L.orc_screen_triangle(hs, len(sketches), screen_val, int(rescue_small), C.byref(ro), C.byref(cols))
    n = len(sketches)
    row_off = np.array([ro[i] for i in range(n + 1)], np.uint64)
    c = np.array([cols[i] for i in range(int(row_off[-1]))], np.uint32)
    L.orc_free_array(ro); L.orc_free_array(cols)
    return row_off, c
