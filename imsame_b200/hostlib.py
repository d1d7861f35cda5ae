"""ctypes view of libimsame_host.so: FASTA ingest, threshold tables, renderer and the
synthetic metagenome generator (host-side C around the GPU hot path)."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.path.join(_HERE, "_lib")
HOST_SO = os.path.join(LIB_DIR, "libimsame_host.so")

_lib = None


class Fasta(C.Structure):
    _fields_ = [("sequences", C.POINTER(C.c_ubyte)), ("start_pos", C.POINTER(C.c_uint64)),
                ("total_len", C.c_uint64), ("n_seqs", C.c_uint64),
                ("break_pos", C.POINTER(C.c_uint64)), ("n_breaks", C.c_uint64)]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(HOST_SO):
            raise RuntimeError(f"{HOST_SO} missing: run `make` (or __graft_entry__.build()) first")
        l = C.CDLL(HOST_SO)
        u8p, u16p, u64p = C.POINTER(C.c_ubyte), C.POINTER(C.c_uint16), C.POINTER(C.c_uint64)
        l.imsame_fasta_load.argtypes = [C.c_char_p, C.c_int, C.POINTER(Fasta)]
        l.imsame_fasta_free.argtypes = [C.POINTER(Fasta)]
        l.imsame_build_nmin.argtypes = [C.c_longdouble, C.c_uint64, u16p]
        l.imsame_build_lmin.argtypes = [C.c_longdouble, u16p]
        l.imsame_build_imin.argtypes = [C.c_longdouble, u16p]
        l.imsame_synth_pool_create.restype = C.c_void_p
        l.imsame_synth_pool_create.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64]
        l.imsame_synth_pool_destroy.argtypes = [C.c_void_p]
        l.imsame_synth_set_threads.argtypes = [C.c_int]
        l.imsame_synth_db_reads.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p]
        l.imsame_synth_query_reads.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32,
                                               C.c_double, C.c_uint32, C.c_void_p]
        l.imsame_synth_write_fasta.argtypes = [C.c_char_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_char]
        l.imsame_format_header.argtypes = [C.c_char_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64]
        l.imsame_render_alignment.restype = C.c_uint64
        l.imsame_render_alignment.argtypes = [C.c_char_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32,
                                              C.c_uint32, C.c_void_p, C.c_uint64]
        _lib = l
    return _lib


def set_synth_threads(n):
    """threads of the synthetic generator (torchrun exports OMP_NUM_THREADS=1)"""
    lib().imsame_synth_set_threads(int(n))


def render_record(read, db_seq, length, identities, x, y, bx, by, ops):
    """header + alignment text of one .align record (src/alignmentFunctions.c:167-168)"""
    x = np.ascontiguousarray(x, dtype=np.uint8)
    y = np.ascontiguousarray(y, dtype=np.uint8)
    ops = np.ascontiguousarray(ops, dtype=np.uint32)
    hdr = C.create_string_buffer(256)
    hl = lib().imsame_format_header(hdr, read, db_seq, length, identities, len(y))
    buf = C.create_string_buffer(6 * (len(x) + len(y)) + 256)
    tl = lib().imsame_render_alignment(buf, x.ctypes.data, len(x), y.ctypes.data, len(y), int(bx), int(by),
                                       ops.ctypes.data, len(ops))
    return hdr.raw[:hl] + buf.raw[:tl]


class SynthPool:
    def __init__(self, seed, n_genomes, genome_len):
        self.h = lib().imsame_synth_pool_create(seed, n_genomes, genome_len)
        if not self.h:
            raise MemoryError("genome pool")
        self.seed = seed

    def db_reads(self, first, count, L, out=None):
        """ASCII reads [first, first+count) of the database stream, shape (count*L,) uint8"""
        if out is None:
            out = np.empty(count * L, dtype=np.uint8)
        lib().imsame_synth_db_reads(self.h, self.seed, first, count, L, out.ctypes.data)
        return out

    def query_reads(self, first, count, L, divergence, n_genomes_used=0, out=None):
        if out is None:
            out = np.empty(count * L, dtype=np.uint8)
        lib().imsame_synth_query_reads(self.h, self.seed, first, count, L, divergence, n_genomes_used,
                                       out.ctypes.data)
        return out

    def close(self):
        if self.h:
            lib().imsame_synth_pool_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()


def write_fasta(path, seq, n_reads, L, prefix):
    rc = lib().imsame_synth_write_fasta(path.encode(), seq.ctypes.data, n_reads, L, prefix.encode())
    if rc:
        raise OSError(path)


def load_fasta(path, is_db):
    """(seq uint8[total], start uint64[n+1], breaks uint64[nb]) as numpy copies"""
    f = Fasta()
    rc = lib().imsame_fasta_load(path.encode(), int(is_db), C.byref(f))
    if rc:
        raise OSError(f"imsame_fasta_load({path}) = {rc}")
    n, ns, nb = int(f.total_len), int(f.n_seqs), int(f.n_breaks)
    seq = np.ctypeslib.as_array(f.sequences, shape=(max(n, 1),))[:n].copy()
    start = np.ctypeslib.as_array(f.start_pos, shape=(ns + 1,)).copy()
    brk = np.ctypeslib.as_array(f.break_pos, shape=(max(nb, 1),))[:nb].copy()
    lib().imsame_fasta_free(C.byref(f))
    return seq, start, brk


def revcomp_is_mirror(text):
    """does the parse of revComp(text) mirror the parse of `text` (bases, read offsets, word breaks)?  The test
    bin/IMSAME_allvsall makes before it derives a reverse-complemented read set on the device."""
    l = lib()
    l.imsame_fasta_parse_mem.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.POINTER(Fasta)]
    l.imsame_revcomp_mem.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
    l.imsame_revcomp_is_mirror.argtypes = [C.POINTER(Fasta), C.POINTER(Fasta)]
    libc = C.CDLL(None)
    libc.free.argtypes = [C.c_void_p]
    fwd, rev, out, n = Fasta(), Fasta(), C.c_void_p(), C.c_size_t()
    if l.imsame_fasta_parse_mem(text, len(text), 1, C.byref(fwd)) or l.imsame_revcomp_mem(text, len(text), C.byref(out), C.byref(n)):
        raise MemoryError("parse / revcomp")
    rc_text = C.string_at(out, n.value)
    libc.free(out)
    if l.imsame_fasta_parse_mem(rc_text, len(rc_text), 1, C.byref(rev)):
        raise MemoryError("parse")
    r = bool(l.imsame_revcomp_is_mirror(C.byref(fwd), C.byref(rev)))
    l.imsame_fasta_free(C.byref(fwd))
    l.imsame_fasta_free(C.byref(rev))
    return r


def threshold_tables(min_e_value, min_coverage, min_identity, db_total_len, max_read=3000):
    nmin = np.zeros(max_read + 1, dtype=np.uint16)
    lmin = np.zeros(max_read + 1, dtype=np.uint16)
    imin = np.zeros(2 * max_read + 1, dtype=np.uint16)
    u16p = C.POINTER(C.c_uint16)
    lib().imsame_build_nmin(C.c_longdouble(min_e_value), db_total_len, nmin.ctypes.data_as(u16p))
    lib().imsame_build_lmin(C.c_longdouble(min_coverage), lmin.ctypes.data_as(u16p))
    lib().imsame_build_imin(C.c_longdouble(min_identity), imin.ctypes.data_as(u16p))
    return nmin, lmin, imin


def sweep_tables(coverages, identities, max_read=3000):
    """imsame_build_sweep_tables: (lmin_sets [n, max_read + 1], imin_sets [n, 2 max_read + 1], lmin_all, imin_all);
    the thresholds pass through double before widening, like make_params"""
    n = len(coverages)
    cov = np.array([float(c) for c in coverages], dtype=np.longdouble)
    idn = np.array([float(i) for i in identities], dtype=np.longdouble)
    lmin_sets = np.zeros((n, max_read + 1), dtype=np.uint16)
    imin_sets = np.zeros((n, 2 * max_read + 1), dtype=np.uint16)
    lmin_all = np.zeros(max_read + 1, dtype=np.uint16)
    imin_all = np.zeros(2 * max_read + 1, dtype=np.uint16)
    l = lib()
    l.imsame_build_sweep_tables.argtypes = [C.c_int] + [C.c_void_p] * 6
    l.imsame_build_sweep_tables.restype = None
    l.imsame_build_sweep_tables(n, cov.ctypes.data, idn.ctypes.data, lmin_sets.ctypes.data, imin_sets.ctypes.data,
                                lmin_all.ctypes.data, imin_all.ctypes.data)
    return lmin_sets, imin_sets, lmin_all, imin_all
