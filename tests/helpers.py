"""Shared test plumbing: ctypes views of the oracle (test infrastructure), the host
library and the reference binary in oracle/_ref (when present)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ORACLE_SO = os.path.join(ROOT, "oracle", "_build", "liboracle.so")
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "IMSAME")
REF_REVCOMP = os.path.join(ROOT, "oracle", "_ref", "revComp")


class OrcSeqs(C.Structure):
    _fields_ = [("seq", C.POINTER(C.c_ubyte)), ("start", C.POINTER(C.c_uint64)),
                ("total_len", C.c_uint64), ("n_seqs", C.c_uint64),
                ("brk", C.POINTER(C.c_uint64)), ("n_brk", C.c_uint64)]


class OrcParams(C.Structure):
    _fields_ = [("min_e_value", C.c_longdouble), ("min_coverage", C.c_longdouble),
                ("min_identity", C.c_longdouble), ("igap", C.c_int), ("egap", C.c_int),
                ("n_threads", C.c_uint64), ("k", C.c_int), ("db_total_len_global", C.c_uint64)]


class OrcBest(C.Structure):
    _fields_ = [("db_seq", C.c_uint64), ("qpos_end", C.c_uint64), ("db_pos", C.c_uint64),
                ("length", C.c_uint32), ("identities", C.c_uint32), ("score", C.c_int32),
                ("bx", C.c_uint32), ("by", C.c_uint32), ("accepted", C.c_uint8)]


class OrcStats(C.Structure):
    _fields_ = [("hits", C.c_uint64), ("evalue_pass", C.c_uint64), ("nw_calls", C.c_uint64),
                ("accepted", C.c_uint64)]


_oracle = None


def build_oracle():
    subprocess.check_call(["make", "-s", "oracle"], cwd=ROOT)


def oracle():
    global _oracle
    if _oracle is None:
        if not os.path.exists(ORACLE_SO):
            build_oracle()
        lib = C.CDLL(ORACLE_SO)
        lib.orc_load_fasta.argtypes = [C.c_char_p, C.c_int, C.POINTER(OrcSeqs)]
        lib.orc_free_seqs.argtypes = [C.POINTER(OrcSeqs)]
        lib.orc_extend.restype = C.c_int64
        lib.orc_extend.argtypes = [C.POINTER(OrcSeqs), C.POINTER(OrcSeqs), C.c_uint64, C.c_uint64,
                                   C.c_uint64, C.c_uint64]
        lib.orc_evalue.restype = C.c_longdouble
        lib.orc_evalue.argtypes = [C.c_int64, C.c_uint64, C.c_uint64]
        lib.orc_default_evalue.restype = C.c_longdouble
        lib.orc_default_evalue.argtypes = []
        u8p = C.POINTER(C.c_ubyte)
        i32p, u32p = C.POINTER(C.c_int32), C.POINTER(C.c_uint32)
        lib.orc_nw_traceback.argtypes = [u8p, C.c_uint64, u8p, C.c_uint64, C.c_int, C.c_int, i32p, u32p,
                                         u32p, u32p, u32p, C.c_char_p, C.c_uint64]
        lib.orc_nw_forward.argtypes = [u8p, C.c_uint64, u8p, C.c_uint64, C.c_int, C.c_int, i32p, u32p,
                                       u32p, u32p, u32p]
        lib.orc_align_sequential.argtypes = [C.POINTER(OrcSeqs), C.POINTER(OrcSeqs), C.POINTER(OrcParams),
                                             C.POINTER(OrcBest), C.c_void_p, C.POINTER(OrcStats)]
        lib.orc_align_bulk.argtypes = [C.POINTER(OrcSeqs), C.POINTER(OrcSeqs), C.POINTER(OrcParams),
                                       C.POINTER(OrcBest), C.POINTER(OrcStats)]
        lib.orc_set_threads.argtypes = [C.c_int]
        lib.orc_set_threads.restype = None
        lib.orc_align_sampled.argtypes = [C.POINTER(OrcSeqs), C.POINTER(OrcSeqs), C.POINTER(OrcParams),
                                          C.POINTER(C.c_uint64), C.c_uint64, C.c_uint64, C.c_uint64,
                                          C.POINTER(OrcBest), C.POINTER(OrcStats)]
        _oracle = lib
    return _oracle


def default_params(n_threads=4, evalue=None, coverage=0.5, identity=0.5, igap=5, egap=2, db_total_len_global=0, k=12):
    """Thresholds exactly as src/IMSAME.c:44-47,552-569 derives them."""
    p = OrcParams()
    if evalue is None:
        p.min_e_value = oracle().orc_default_evalue()  # 1/powl(10,20) evaluated in long double (src/IMSAME.c:44)
    else:
        p.min_e_value = float(evalue)
    p.min_coverage = float(coverage)
    p.min_identity = float(identity)
    p.igap = -int(igap)
    p.egap = -int(egap)
    p.n_threads = n_threads
    p.k = k  # 12 = FIXED_K (src/structs.h:15), the only value the reference itself can pin
    p.db_total_len_global = db_total_len_global
    return p


class OracleSeqs:
    """Owns an orc_seqs loaded from FASTA or built from numpy arrays."""

    def __init__(self, path=None, is_db=False, seq=None, start=None, brk=None):
        self.s = OrcSeqs()
        self._own = False
        if path is not None:
            rc = oracle().orc_load_fasta(path.encode(), int(is_db), C.byref(self.s))
            assert rc == 0, rc
            self._own = True
        else:
            self._seq = np.ascontiguousarray(seq, dtype=np.uint8)
            st = np.asarray(start, dtype=np.uint64)
            if len(st) == 0 or st[-1] != len(self._seq):
                st = np.concatenate([st, np.array([len(self._seq)], dtype=np.uint64)])
            self._start = np.ascontiguousarray(st)
            self._brk = np.ascontiguousarray(brk if brk is not None else [], dtype=np.uint64)
            self.s.seq = self._seq.ctypes.data_as(C.POINTER(C.c_ubyte))
            self.s.start = self._start.ctypes.data_as(C.POINTER(C.c_uint64))
            self.s.total_len = len(self._seq)
            self.s.n_seqs = len(self._start) - 1
            self.s.brk = self._brk.ctypes.data_as(C.POINTER(C.c_uint64))
            self.s.n_brk = len(self._brk)

    def numpy(self):
        n = int(self.s.total_len)
        seq = np.ctypeslib.as_array(self.s.seq, shape=(max(n, 1),))[:n]
        start = np.ctypeslib.as_array(self.s.start, shape=(int(self.s.n_seqs) + 1,))
        nb = int(self.s.n_brk)
        brk = np.ctypeslib.as_array(self.s.brk, shape=(max(nb, 1),))[:nb]
        return seq, start, brk

    def __del__(self):
        if self._own:
            try:
                oracle().orc_free_seqs(C.byref(self.s))
            except Exception:
                pass


def oracle_align(db, q, params, bulk=False, out_path=None):
    lib = oracle()
    nq = int(q.s.n_seqs)
    best = (OrcBest * max(nq, 1))()
    st = OrcStats()
    if bulk:
        rc = lib.orc_align_bulk(C.byref(db.s), C.byref(q.s), C.byref(params), best, C.byref(st))
    else:
        fp = None
        libc = C.CDLL(None)
        libc.fopen.restype = C.c_void_p
        libc.fclose.argtypes = [C.c_void_p]
        if out_path:
            fp = libc.fopen(out_path.encode(), b"wb")
        rc = lib.orc_align_sequential(C.byref(db.s), C.byref(q.s), C.byref(params), best, fp, C.byref(st))
        if fp:
            libc.fclose(fp)
    assert rc == 0, rc
    return best, st


def oracle_set_threads(n):
    oracle().orc_set_threads(int(n))


def oracle_align_sampled(db, q, params, reads, db_pos_base=0, db_seq_base=0):
    """index-free per-read checker (oracle/imsame_sampled.c): first accepted hit of the query reads
    `reads` against db (whole database or one shard).  Returns ({read: (db_seq, qpos_end, db_pos, length,
    identities)} for the accepted ones, stats)."""
    reads = np.ascontiguousarray(reads, dtype=np.uint64)
    n = len(reads)
    best = (OrcBest * max(n, 1))()
    st = OrcStats()
    rc = oracle().orc_align_sampled(C.byref(db.s), C.byref(q.s), C.byref(params),
                                    reads.ctypes.data_as(C.POINTER(C.c_uint64)), n, int(db_pos_base),
                                    int(db_seq_base), best, C.byref(st))
    assert rc == 0, rc
    rec = {int(reads[i]): (best[i].db_seq, best[i].qpos_end, best[i].db_pos, best[i].length, best[i].identities)
           for i in range(n) if best[i].accepted}
    return rec, st


def best_to_records(best, nq):
    """{read: (db_seq, qpos_end, db_pos, length, identities)} for accepted reads"""
    return {r: (best[r].db_seq, best[r].qpos_end, best[r].db_pos, best[r].length, best[r].identities)
            for r in range(nq) if best[r].accepted}


HEADER_RE = re.compile(rb"^\((\d+), (\d+)\) : (\d+)% (\d+)% (\d+)$")


def parse_align_headers(path):
    """sorted list of (read, db_seq, id%, cov%, ylen) from a .align file"""
    out = []
    with open(path, "rb") as f:
        for line in f:
            if line.startswith(b"("):
                m = HEADER_RE.match(line.rstrip(b"\n"))
                if m:
                    out.append(tuple(int(x) for x in m.groups()))
    return sorted(out)


def split_align_records(path):
    """{(read, db_seq): full record bytes} -- order-insensitive comparison of whole files"""
    recs = {}
    cur_key, cur = None, []
    with open(path, "rb") as f:
        for line in f:
            m = HEADER_RE.match(line.rstrip(b"\n")) if line.startswith(b"(") else None
            if m:
                if cur_key is not None:
                    recs[cur_key] = b"".join(cur)
                cur_key, cur = (int(m.group(1)), int(m.group(2))), [line]
            else:
                cur.append(line)
    if cur_key is not None:
        recs[cur_key] = b"".join(cur)
    return recs


def have_reference():
    return os.path.exists(REF_BIN)


PINS = os.path.join(ROOT, "tests", "golden", "reference_pins.json")
_pins = None


def pins(section):
    """what the reference tools gave on the seeded inputs of the tests that compare with them (see the file's "about")"""
    global _pins
    if _pins is None:
        import json
        with open(PINS) as f:
            _pins = json.load(f)
    return _pins[section]


def sha(data):
    import hashlib
    return hashlib.sha256(data).hexdigest()


def align_digest(path, whole=False, lines=False):
    """the parts of a .align file the reference comparisons look at: record count, sorted header lines, the sorted
    lines of the whole file (lines=True), the bytes (whole=True: -n_threads 1 output)"""
    data = open(path, "rb").read()
    d = {"records": len(parse_align_headers(path)),
         "headers": sha(b"\n".join(sorted(l for l in data.split(b"\n") if HEADER_RE.match(l))))}
    if lines:
        d["sorted_lines"] = sha(b"\n".join(sorted(data.split(b"\n"))))
    if whole:
        d["bytes"] = sha(data)
    return d


def run_reference(query_fa, db_fa, out_path, n_threads=4, extra=()):
    """Run the unmodified reference binary; returns its stdout."""
    cmd = [REF_BIN, "-query", query_fa, "-db", db_fa, "-out", out_path, "-n_threads", str(n_threads)]
    cmd += list(extra)
    return subprocess.run(cmd, check=True, capture_output=True, text=True).stdout


def header_tuple(read, db_seq, length, identities, ylen):
    return (read, db_seq, min(100, 100 * identities // length), min(100, 100 * length // ylen), ylen)
