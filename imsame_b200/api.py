"""ctypes binding of the C ABI in include/imsame_gpu.h (libimsame_gpu.so).

This is the Python-side stub a maintainer would write against the C ABI; it holds no
algorithm.  The argument names follow the reference's HashTableArgs
(src/alignmentFunctions.h:10-30): database / query SeqInfo, min_e_value, min_coverage,
min_identity, igap, egap (negated), and -n_threads (src/IMSAME.c:414,433).

There is deliberately no fallback: if the CUDA library is missing or no sm_100 device
is present, construction raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
GPU_SO = os.environ.get("IMSAME_GPU_SO") or os.path.join(_HERE, "_lib", "libimsame_gpu.so")  # override: experiments

KEY_NONE = 0x7FFFFFFFFFFFFFFF
SWEEP_MAX = 16  # IMSAME_SWEEP_MAX


class SeqInfo(C.Structure):
    _fields_ = [("sequences", C.c_void_p), ("start_pos", C.c_void_p), ("total_len", C.c_uint64),
                ("n_seqs", C.c_uint64), ("break_pos", C.c_void_p), ("n_breaks", C.c_uint64)]


class Params(C.Structure):
    _fields_ = [("min_e_value", C.c_longdouble), ("min_coverage", C.c_longdouble),
                ("min_identity", C.c_longdouble), ("igap", C.c_int), ("egap", C.c_int),
                ("n_threads", C.c_uint64), ("db_total_len_global", C.c_uint64),
                ("db_pos_base", C.c_uint64), ("db_seq_base", C.c_uint64)]


class Best(C.Structure):
    _fields_ = [("db_seq", C.c_uint64), ("qpos_end", C.c_uint64), ("db_pos", C.c_uint64),
                ("length", C.c_uint32), ("identities", C.c_uint32), ("accepted", C.c_uint32),
                ("reserved", C.c_uint32)]


BEST_DTYPE = np.dtype([("db_seq", "<u8"), ("qpos_end", "<u8"), ("db_pos", "<u8"), ("length", "<u4"),
                       ("identities", "<u4"), ("accepted", "<u4"), ("reserved", "<u4")])


class Stats(C.Structure):
    _fields_ = [("n_query_kmers", C.c_uint64), ("n_db_kmers", C.c_uint64), ("n_hits", C.c_uint64),
                ("n_evalue_pass", C.c_uint64), ("n_pairs", C.c_uint64), ("n_pairs_dp", C.c_uint64),
                ("n_cells", C.c_uint64), ("n_accepted", C.c_uint64),
                ("ms_pack_query", C.c_float), ("ms_k1", C.c_float), ("ms_pack_db", C.c_float),
                ("ms_k2", C.c_float), ("ms_k2b", C.c_float), ("ms_k3", C.c_float), ("ms_select", C.c_float),
                ("ms_h2d", C.c_float), ("ms_d2h", C.c_float), ("ms_total", C.c_float),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("k2_launches", C.c_uint32), ("k3_launches", C.c_uint32), ("total_launches", C.c_uint32),
                ("k3_packed_launches", C.c_uint32), ("ms_comm", C.c_float), ("scan_passes", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved"}


# every symbol declared in include/imsame_gpu.h
SYMBOLS = ["imsame_gpu_create", "imsame_gpu_destroy", "imsame_gpu_strerror", "imsame_gpu_last_cuda_error", "imsame_gpu_mem_info",
           "imsame_gpu_set_stream", "imsame_gpu_align", "imsame_gpu_set_query", "imsame_gpu_set_db",
           "imsame_gpu_run", "imsame_gpu_n_segments", "imsame_gpu_n_bands", "imsame_gpu_run_begin",
           "imsame_gpu_run_scan", "imsame_gpu_run_band", "imsame_gpu_run_select", "imsame_gpu_run_end",
           "imsame_gpu_mask_payload", "imsame_gpu_fetch", "imsame_gpu_nw_batch", "imsame_gpu_set_nw_mode", "imsame_gpu_set_passes",
           "imsame_gpu_set_kmer", "imsame_gpu_comm_id", "imsame_gpu_comm_init", "imsame_gpu_comm_free",
           "imsame_gpu_run_sharded", "imsame_gpu_align_shard", "imsame_gpu_align_sharded",
           "imsame_gpu_db_revcomp", "imsame_gpu_align_revcomp", "imsame_gpu_align_sweep",
           "imsame_gpu_sample_create", "imsame_gpu_sample_revcomp", "imsame_gpu_sample_free", "imsame_gpu_align_samples",
           "imsame_gpu_traceback", "imsame_gpu_free", "imsame_gpu_host_alloc", "imsame_gpu_host_free"]

_lib = None


class ImsameError(RuntimeError):
    def __init__(self, code, detail=""):
        self.code = code
        msg = lib().imsame_gpu_strerror(code).decode()
        super().__init__(f"imsame_gpu error {code}: {msg}" + (f" [{detail}]" if detail else ""))


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(GPU_SO):
            raise RuntimeError(f"{GPU_SO} missing: the CUDA extension is required (no CPU fallback); "
                               f"run `make` or __graft_entry__.build()")
        l = C.CDLL(GPU_SO)
        vp, u64 = C.c_void_p, C.c_uint64
        l.imsame_gpu_create.argtypes = [C.POINTER(vp), C.c_int]
        l.imsame_gpu_destroy.argtypes = [vp]
        l.imsame_gpu_destroy.restype = None
        l.imsame_gpu_strerror.argtypes = [C.c_int]
        l.imsame_gpu_strerror.restype = C.c_char_p
        l.imsame_gpu_last_cuda_error.argtypes = [vp]
        l.imsame_gpu_last_cuda_error.restype = C.c_char_p
        l.imsame_gpu_mem_info.argtypes = [vp, C.POINTER(u64), C.POINTER(u64)]
        l.imsame_gpu_set_stream.argtypes = [vp, vp]
        l.imsame_gpu_align.argtypes = [vp, C.POINTER(SeqInfo), C.POINTER(SeqInfo), C.POINTER(Params), vp,
                                       C.POINTER(Stats)]
        l.imsame_gpu_align_sweep.argtypes = [vp, C.POINTER(SeqInfo), C.POINTER(SeqInfo), vp, C.c_int, vp, vp,
                                             C.POINTER(Stats)]
        l.imsame_gpu_set_query.argtypes = [vp, C.POINTER(SeqInfo), C.POINTER(Params)]
        l.imsame_gpu_set_db.argtypes = [vp, C.POINTER(SeqInfo)]
        l.imsame_gpu_run.argtypes = [vp, C.POINTER(Params), vp, vp, C.POINTER(Stats)]
        l.imsame_gpu_n_segments.argtypes = [vp]
        l.imsame_gpu_run_begin.argtypes = [vp, C.POINTER(Params), vp, vp]
        l.imsame_gpu_run_scan.argtypes = [vp, C.c_int]
        l.imsame_gpu_run_band.argtypes = [vp, C.c_int, C.c_int]
        l.imsame_gpu_run_select.argtypes = [vp, C.c_int]
        l.imsame_gpu_run_end.argtypes = [vp, C.POINTER(Stats)]
        l.imsame_gpu_mask_payload.argtypes = [vp, vp, vp, vp]
        l.imsame_gpu_fetch.argtypes = [vp, vp, vp, vp]
        l.imsame_gpu_nw_batch.argtypes = [vp, C.c_uint32, vp, vp, vp, vp, C.c_int, C.c_int, vp,
                                          C.POINTER(C.c_float)]
        l.imsame_gpu_traceback.argtypes = [vp, C.POINTER(SeqInfo), C.POINTER(SeqInfo), C.POINTER(Params), vp, vp,
                                           C.POINTER(C.POINTER(C.c_uint32)), vp]
        l.imsame_gpu_set_nw_mode.argtypes = [vp, C.c_int]
        l.imsame_gpu_set_passes.argtypes = [vp, C.c_int]
        l.imsame_gpu_set_kmer.argtypes = [vp, C.c_int]
        l.imsame_gpu_comm_id.argtypes = [vp]
        l.imsame_gpu_comm_init.argtypes = [vp, vp, C.c_int, C.c_int]
        l.imsame_gpu_comm_free.argtypes = [vp]
        l.imsame_gpu_run_sharded.argtypes = [vp, C.POINTER(Params), vp, vp, C.c_int, C.POINTER(Stats)]
        l.imsame_gpu_align_shard.argtypes = [vp, C.POINTER(SeqInfo), C.POINTER(SeqInfo), C.POINTER(Params), vp, vp, C.POINTER(Stats)]
        l.imsame_gpu_align_sharded.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(SeqInfo), C.POINTER(SeqInfo),
                                               C.POINTER(Params), vp, C.POINTER(Stats)]
        l.imsame_gpu_db_revcomp.argtypes = [vp]
        l.imsame_gpu_align_revcomp.argtypes = [C.POINTER(vp), C.c_int, vp, C.POINTER(Stats)]
        l.imsame_gpu_sample_create.argtypes = [vp, C.POINTER(SeqInfo), C.POINTER(vp)]
        l.imsame_gpu_sample_revcomp.argtypes = [vp, vp, C.POINTER(vp)]
        l.imsame_gpu_sample_free.argtypes = [vp, vp]
        l.imsame_gpu_sample_free.restype = None
        l.imsame_gpu_align_samples.argtypes = [vp, vp, vp, C.POINTER(Params), vp, C.POINTER(Stats)]
        l.imsame_gpu_free.argtypes = [vp]
        l.imsame_gpu_free.restype = None
        l.imsame_gpu_host_alloc.argtypes = [u64]
        l.imsame_gpu_host_alloc.restype = vp
        l.imsame_gpu_host_free.argtypes = [vp]
        l.imsame_gpu_host_free.restype = None
        _lib = l
    return _lib


def make_params(min_e_value=None, min_coverage=0.5, min_identity=0.5, igap=5, egap=2, n_threads=4,
                db_total_len_global=0, db_pos_base=0, db_seq_base=0):
    """Defaults and conversions of src/IMSAME.c:44-49,552-569 (igap/egap given positive, stored negated;
    thresholds pass through double before widening; the default e-value is 1/powl(10,20))."""
    p = Params()
    if min_e_value is None:
        p.min_e_value = default_evalue()
    else:
        p.min_e_value = float(min_e_value)
    p.min_coverage = float(min_coverage)
    p.min_identity = float(min_identity)
    p.igap = -int(igap)
    p.egap = -int(egap)
    p.n_threads = int(n_threads)
    p.db_total_len_global = int(db_total_len_global)
    p.db_pos_base = int(db_pos_base)
    p.db_seq_base = int(db_seq_base)
    return p


def default_evalue():
    """1/powl(10, 20) in long double, src/IMSAME.c:44 (numpy longdouble is the x87 type on x86-64)."""
    ten = np.longdouble(10)
    v = np.longdouble(1) / (ten ** 20)
    return C.c_longdouble.from_buffer_copy(np.asarray(v, dtype=np.longdouble).tobytes()).value


class PinnedArray:
    """uint8/uint64 numpy view over cudaHostAlloc'ed memory (full-speed H2D copies)."""

    def __init__(self, n, dtype=np.uint8):
        self.nbytes = int(n) * np.dtype(dtype).itemsize
        self.ptr = lib().imsame_gpu_host_alloc(self.nbytes)
        if not self.ptr:
            raise MemoryError("cudaHostAlloc")
        buf = (C.c_ubyte * self.nbytes).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(n))

    def free(self):
        if self.ptr:
            self.array = None
            lib().imsame_gpu_host_free(self.ptr)
            self.ptr = None


def _seqinfo(seq, start, breaks=None):
    """seq: uint8 ASCII; start: uint64 offsets (n or n+1 entries)"""
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    start = np.ascontiguousarray(start, dtype=np.uint64)
    n = len(start)
    if n >= 2 and int(start[-1]) == len(seq):
        n -= 1  # n+1 form (sentinel = total_len); an n-form cannot end there: empty reads are not allowed
    s = SeqInfo()
    s.sequences = seq.ctypes.data
    s.start_pos = start.ctypes.data
    s.total_len = len(seq)
    s.n_seqs = n
    keep = [seq, start]
    if breaks is not None and len(breaks):
        b = np.ascontiguousarray(breaks, dtype=np.uint64)
        s.break_pos = b.ctypes.data
        s.n_breaks = len(b)
        keep.append(b)
    return s, keep


class Imsame:
    """One GPU context (one process per GPU)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        rc = lib().imsame_gpu_create(C.byref(self._h), device)
        if rc:
            raise ImsameError(rc)
        self.nq = 0

    def close(self):
        if self._h:
            lib().imsame_gpu_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc:
            raise ImsameError(rc, lib().imsame_gpu_last_cuda_error(self._h).decode())

    def set_stream(self, cuda_stream_ptr):
        """run all work of this context on an existing stream.  torch's default stream has the raw handle 0,
        which the C ABI reads as "use your own stream": it is passed as cudaStreamLegacy (handle 1) instead, so
        that the library's kernels and torch / NCCL operations issued on the default stream stay ordered."""
        self._check(lib().imsame_gpu_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 1)))

    # -- one call: index + scan + NW + selection (src/IMSAME.c:232-281 + :409-467)
    def set_nw_mode(self, mode):
        """0 = packed-word K3 where eligible (default), 1 = generic K3 only"""
        self._check(lib().imsame_gpu_set_nw_mode(self._h, int(mode)))

    def set_passes(self, mode):
        """0 = decide per run (default), 1 = one scan with every word, 2 = early words first (two scans)"""
        self._check(lib().imsame_gpu_set_passes(self._h, int(mode)))

    def set_kmer(self, k):
        """seed length, 4..16 (default 12 = the reference's FIXED_K); call before set_query / align"""
        self._check(lib().imsame_gpu_set_kmer(self._h, int(k)))

    def align(self, db, query, params=None, db_breaks=None):
        """db, query: (seq uint8 ASCII, start uint64[n+1]). Returns (records ndarray BEST_DTYPE, stats dict)."""
        params = params or make_params()
        d, k1 = _seqinfo(db[0], db[1], db_breaks)
        q, k2 = _seqinfo(query[0], query[1])
        out = np.zeros(int(q.n_seqs), dtype=BEST_DTYPE)
        st = Stats()
        self._check(lib().imsame_gpu_align(self._h, C.byref(d), C.byref(q), C.byref(params), out.ctypes.data,
                                           C.byref(st)))
        self.nq = int(q.n_seqs)
        return out, st.as_dict()

    def align_sweep(self, db, query, params_list, db_breaks=None):
        """one run, several coverage/identity sets (imsame_gpu_align_sweep): params_list = Params that differ only in
        min_coverage / min_identity (at most SWEEP_MAX).  Returns ([records per set], [IMSAME_OK or IMSAME_EREADSIZE
        per set], stats): set t's records are what align() with params_list[t] returns; a set whose code is not 0
        has all-zero records."""
        d, k1 = _seqinfo(db[0], db[1], db_breaks)
        q, k2 = _seqinfo(query[0], query[1])
        n, nq = len(params_list), int(q.n_seqs)
        ps = (Params * max(n, 1))(*params_list)
        out = np.zeros(max(n, 1) * nq, dtype=BEST_DTYPE)
        codes = np.zeros(max(n, 1), dtype=np.int32)
        st = Stats()
        self._check(lib().imsame_gpu_align_sweep(self._h, C.byref(d), C.byref(q), C.cast(ps, C.c_void_p), n,
                                                 out.ctypes.data, codes.ctypes.data, C.byref(st)))
        self.nq = nq
        return [out[t * nq:(t + 1) * nq].copy() for t in range(n)], [int(c) for c in codes[:n]], st.as_dict()

    # -- staged form
    def set_query(self, query, params=None):
        params = params or make_params()
        q, keep = _seqinfo(query[0], query[1])
        self._check(lib().imsame_gpu_set_query(self._h, C.byref(q), C.byref(params)))
        self.nq = int(q.n_seqs)

    def set_db(self, db, db_breaks=None):
        d, keep = _seqinfo(db[0], db[1], db_breaks)
        self._check(lib().imsame_gpu_set_db(self._h, C.byref(d)))

    def run(self, params=None, d_keys=0, d_payload=0):
        params = params or make_params()
        st = Stats()
        self._check(lib().imsame_gpu_run(self._h, C.byref(params), C.c_void_p(d_keys), C.c_void_p(d_payload),
                                         C.byref(st)))
        return st.as_dict()

    def run_stepped(self, params=None, d_keys=0, d_payload=0, exchange=None, exchange_every=1):
        """imsame_gpu_run in steps; `exchange()` is called between bands (multi-GPU: all-reduce MIN of the
        keys), every `exchange_every` bands and after the last band of each segment."""
        params = params or make_params()
        L = lib()
        self._check(L.imsame_gpu_run_begin(self._h, C.byref(params), C.c_void_p(d_keys), C.c_void_p(d_payload)))
        nb, nseg = L.imsame_gpu_n_bands(), L.imsame_gpu_n_segments(self._h)
        for seg in range(nseg):
            self._check(L.imsame_gpu_run_scan(self._h, seg))
        for band in range(nb):  # band-major over all segments: global scan order of the candidates
            for seg in range(nseg):
                self._check(L.imsame_gpu_run_band(self._h, seg, band))
            if exchange is not None and ((band + 1) % exchange_every == 0 or band == nb - 1):
                exchange()
        for seg in range(nseg):
            self._check(L.imsame_gpu_run_select(self._h, seg))
        st = Stats()
        self._check(L.imsame_gpu_run_end(self._h, C.byref(st)))
        return st.as_dict()

    # -- the reverse strand of the resident database
    def db_revcomp(self):
        """the resident database becomes its reverse complement (reads in reverse order, each reverse complemented:
        what revComp writes); a second call restores it"""
        self._check(lib().imsame_gpu_db_revcomp(self._h))

    def align_revcomp(self):
        """the query and parameters of the previous align(), against the reverse complement of its database, which is
        still resident.  Returns (records, stats) like align(); db_seq / db_pos count in the reverse database."""
        out, st = align_revcomp([self])
        return out, st[0]

    # -- read sets resident on the device (all-vs-all)
    def sample(self, reads, breaks=None):
        """upload + pack once; returns a handle usable as database or query of align_samples"""
        d, keep = _seqinfo(reads[0], reads[1], breaks)
        h = C.c_void_p()
        self._check(lib().imsame_gpu_sample_create(self._h, C.byref(d), C.byref(h)))
        return Sample(self, h, int(d.n_seqs))

    def sample_revcomp(self, sample):
        """reverse complement on the device, records in reverse order (what revComp writes)"""
        h = C.c_void_p()
        self._check(lib().imsame_gpu_sample_revcomp(self._h, sample._h, C.byref(h)))
        return Sample(self, h, sample.n)

    def align_samples(self, db, query, params=None):
        params = params or make_params()
        out = np.zeros(query.n, dtype=BEST_DTYPE)
        st = Stats()
        self._check(lib().imsame_gpu_align_samples(self._h, db._h, query._h, C.byref(params), out.ctypes.data, C.byref(st)))
        self.nq = query.n
        return out, st.as_dict()

    # -- database sharded over several GPUs, reduced by NCCL inside the library
    def comm_init(self, comm_id, n_ranks, rank):
        """join the communicator named by the 128 bytes rank 0 obtained from comm_id()"""
        buf = (C.c_ubyte * COMM_ID_BYTES).from_buffer_copy(bytes(comm_id))
        self._check(lib().imsame_gpu_comm_init(self._h, C.cast(buf, C.c_void_p), int(n_ranks), int(rank)))

    def comm_free(self):
        self._check(lib().imsame_gpu_comm_free(self._h))

    def run_sharded(self, params, d_keys=0, d_payload=0, exchange_every=0):
        """collective: scan + NW over this rank's shard with ncclMin key reductions between bands and the
        owner's payload (ncclMax) at the end; d_keys / d_payload hold the reduced result on every rank"""
        st = Stats()
        self._check(lib().imsame_gpu_run_sharded(self._h, C.byref(params), C.c_void_p(d_keys), C.c_void_p(d_payload),
                                                 int(exchange_every), C.byref(st)))
        return st.as_dict()

    def align_shard(self, shard, query, params, d_keys=0, d_payload=0, db_breaks=None):
        """collective, host buffers in: query + this rank's shard uploaded (segments one ahead of their scan), then as
        run_sharded.  The reduced result stays on the device (d_keys / d_payload or the context's own): fetch() it."""
        d, k1 = _seqinfo(shard[0], shard[1], db_breaks)
        q, k2 = _seqinfo(query[0], query[1])
        st = Stats()
        self._check(lib().imsame_gpu_align_shard(self._h, C.byref(d), C.byref(q), C.byref(params), C.c_void_p(d_keys),
                                                 C.c_void_p(d_payload), C.byref(st)))
        self.nq = int(q.n_seqs)
        return st.as_dict()

    def n_segments(self):
        return lib().imsame_gpu_n_segments(self._h)

    def mask_payload(self, d_keys_reduced, d_keys_local, d_payload):
        self._check(lib().imsame_gpu_mask_payload(self._h, C.c_void_p(d_keys_reduced), C.c_void_p(d_keys_local),
                                                  C.c_void_p(d_payload)))

    def fetch(self, d_keys=0, d_payload=0):
        out = np.zeros(self.nq, dtype=BEST_DTYPE)
        self._check(lib().imsame_gpu_fetch(self._h, C.c_void_p(d_keys), C.c_void_p(d_payload), out.ctypes.data))
        return out

    # -- winners-only traceback (device) + text (host/render.c): the body of the .align records
    def traceback(self, db, query, best, params=None, db_breaks=None):
        """returns (ops_off uint64[nq+1], ops uint32[], cell_xy uint32[nq,4])"""
        params = params or make_params()
        d, k1 = _seqinfo(db[0], db[1], db_breaks)
        q, k2 = _seqinfo(query[0], query[1])
        nq = int(q.n_seqs)
        best = np.ascontiguousarray(best, dtype=BEST_DTYPE)
        ops_off = np.zeros(nq + 1, dtype=np.uint64)
        cell = np.zeros((nq, 4), dtype=np.uint32)
        ops_p = C.POINTER(C.c_uint32)()
        self._check(lib().imsame_gpu_traceback(self._h, C.byref(d), C.byref(q), C.byref(params), best.ctypes.data,
                                               ops_off.ctypes.data, C.byref(ops_p), cell.ctypes.data))
        n = int(ops_off[nq])
        ops = np.ctypeslib.as_array(ops_p, shape=(max(n, 1),))[:n].copy()
        lib().imsame_gpu_free(C.cast(ops_p, C.c_void_p))
        return ops_off, ops, cell

    # -- NW on explicit pairs
    def nw_batch(self, xs, ys, igap=5, egap=2):
        """xs, ys: lists of ASCII byte strings / uint8 arrays. Returns (int32[n,5], kernel ms):
        score, bx, by, length, identities."""
        n = len(xs)
        xa = [np.ascontiguousarray(np.frombuffer(x, dtype=np.uint8) if isinstance(x, (bytes, bytearray)) else x,
                                   dtype=np.uint8) for x in xs]
        ya = [np.ascontiguousarray(np.frombuffer(y, dtype=np.uint8) if isinstance(y, (bytes, bytearray)) else y,
                                   dtype=np.uint8) for y in ys]
        xp = (C.c_void_p * n)(*[a.ctypes.data for a in xa])
        yp = (C.c_void_p * n)(*[a.ctypes.data for a in ya])
        xl = np.array([len(a) for a in xa], dtype=np.uint32)
        yl = np.array([len(a) for a in ya], dtype=np.uint32)
        out = np.zeros((n, 5), dtype=np.int32)
        ms = C.c_float(0)
        self._check(lib().imsame_gpu_nw_batch(self._h, n, C.cast(xp, C.c_void_p), xl.ctypes.data,
                                              C.cast(yp, C.c_void_p), yl.ctypes.data, -int(igap), -int(egap),
                                              out.ctypes.data, C.byref(ms)))
        return out, ms.value


class Sample:
    """a read set resident on the device (imsame_gpu_sample_*)"""

    def __init__(self, ctx, handle, n):
        self.ctx, self._h, self.n = ctx, handle, n

    def free(self):
        if self._h:
            lib().imsame_gpu_sample_free(self.ctx._h, self._h)
            self._h = C.c_void_p()


COMM_ID_BYTES = 128


def comm_id():
    """128 opaque bytes naming a new communicator (ncclGetUniqueId); hand them to every rank"""
    buf = (C.c_ubyte * COMM_ID_BYTES)()
    rc = lib().imsame_gpu_comm_id(C.cast(buf, C.c_void_p))
    if rc:
        raise ImsameError(rc)
    return bytes(buf)


def align_sharded(ctxs, db, query, params=None, db_breaks=None):
    """one process, len(ctxs) GPUs: imsame_gpu_align_sharded.  Returns (records, [stats per shard])."""
    params = params or make_params()
    d, k1 = _seqinfo(db[0], db[1], db_breaks)
    q, k2 = _seqinfo(query[0], query[1])
    n = len(ctxs)
    out = np.zeros(int(q.n_seqs), dtype=BEST_DTYPE)
    hs = (C.c_void_p * n)(*[c._h for c in ctxs])
    st = (Stats * n)()
    rc = lib().imsame_gpu_align_sharded(hs, n, C.byref(d), C.byref(q), C.byref(params), out.ctypes.data, st)
    if rc:
        raise ImsameError(rc, lib().imsame_gpu_last_cuda_error(ctxs[0]._h).decode())
    for c in ctxs:
        c.nq = int(q.n_seqs)
    return out, [s.as_dict() for s in st]


def align_revcomp(ctxs):
    """one process, len(ctxs) GPUs: the previous align_sharded() (or, one context, align()) again, against the reverse
    complement of its database, still resident on the same contexts.  Returns (records, [stats per shard])."""
    n = len(ctxs)
    out = np.zeros(ctxs[0].nq, dtype=BEST_DTYPE)
    hs = (C.c_void_p * n)(*[c._h for c in ctxs])
    st = (Stats * n)()
    rc = lib().imsame_gpu_align_revcomp(hs, n, out.ctypes.data, st)
    if rc:
        raise ImsameError(rc, lib().imsame_gpu_last_cuda_error(ctxs[0]._h).decode())
    return out, [s.as_dict() for s in st]


def header_fields(read, rec, ylen):
    """(read, db_seq, id%, cov%, ylen) exactly as printed at src/alignmentFunctions.c:167"""
    length, ident = int(rec["length"]), int(rec["identities"])
    return (int(read), int(rec["db_seq"]), min(100, 100 * ident // length), min(100, 100 * length // ylen),
            int(ylen))
