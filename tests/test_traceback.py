"""The alignment of accepted hits (imsame_gpu_align_traceback, IMSAME / IMSAME_allvsall -cigar): CIGAR, exact
coordinates and counts computed on the GPU (csrc/cigar.cuh), checked by replaying every CIGAR over its two reads and
against a plain Python NW with traceback that follows the documented tie-breaking (so the CIGARs must be identical).
CPU: the kernel's device functions stepped as a warp (tests/emul/cigar_emul.cpp), the Python reference against the
oracle's forward NW.  GPU: random and golden inputs, edge cases, batch splitting, reverse strand, sweeps, command lines."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as hp
import synth_cases as sc

G = os.path.join(hp.ROOT, "tests", "golden")
EXE = os.path.join(hp.ROOT, "bin", "IMSAME")
ALLVSALL = os.path.join(hp.ROOT, "bin", "IMSAME_allvsall")
REVCOMP = os.path.join(hp.ROOT, "bin", "revComp")
COLS_RE = re.compile(rb"^\((\d+), (\d+)\) : (\d+)% (\d+)% (\d+) (\d+) (\d+) (\d+) (\d+) (-?\d+) ((?:\d+[=XID])+)$")
CIGAR_RE = re.compile(r"(\d+)([=XID])")
COMP = np.arange(256, dtype=np.uint8)
for _a, _b in zip(b"ACGT", b"TGCA"):
    COMP[_a] = _b


# ---- reference: the reference's NW (src/alignmentFunctions.c:389-489) with back-pointers, in plain Python ----------
def ref_nw(x, y, igap, egap):
    """x = database read, y = query read (bytes); igap / egap as stored (negated).  Tie-breaking as documented in
    csrc/cigar.cuh.  Returns (score, bx, by, cigar text, (db_start, q_start))."""
    P, NEG = 4, -(1 << 60)
    X, Y = len(x), len(y)
    T = [[0] * Y for _ in range(X)]
    F = [[None] * Y for _ in range(X)]  # (kind, from_x, from_y)
    mcs = [P if x[0] == y[j] else -P for j in range(Y)]
    mcx = [0] * Y
    for j in range(Y):
        T[0][j] = mcs[j]
    best = (NEG, 0, 0)
    for i in range(1, X):
        Ti, Tp = T[i], T[i - 1]
        Ti[0] = P if x[i] == y[0] else -P
        mfs, mfy = Ti[0], 0
        for j in range(1, Y):
            if j > 1 and mfs <= Ti[j - 2]:
                mfs, mfy = Tp[j - 2], j - 2
            m = P if x[i] == y[j] else -P
            d = Tp[j - 1] + m
            l = mfs + igap + (j - mfy - 1) * egap + m if j > 1 else NEG
            r = mcs[j - 1] + igap + (i - mcx[j - 1] - 1) * egap + m if i > 1 else NEG
            if d >= l and d >= r:
                Ti[j], F[i][j] = d, ("M", i - 1, j - 1)
            elif r > l:
                Ti[j], F[i][j] = r, ("D", mcx[j - 1], j - 1)
            else:
                Ti[j], F[i][j] = l, ("I", i - 1, mfy)
            if i > 1 and j > 1 and T[i - 2][j - 1] > mcs[j - 1]:
                mcs[j - 1], mcx[j - 1] = T[i - 2][j - 1], i - 2
            if (i == X - 1 or j == Y - 1) and Ti[j] >= best[0]:
                best = (Ti[j], i, j)
    s, bx, by = best
    cols, px, py = [], bx, by
    cols.append("=" if x[px] == y[py] else "X")
    while px > 0 and py > 0:
        kind, ux, uy = F[px][py]
        if kind == "D":
            cols += ["D"] * (px - ux - 1)
        elif kind == "I":
            cols += ["I"] * (py - uy - 1)
        px, py = ux, uy
        cols.append("=" if x[px] == y[py] else "X")
    return s, bx, by, runs_text(cols[::-1]), (px, py)


def runs_text(cols):
    out, k = [], 0
    while k < len(cols):
        e = k
        while e < len(cols) and cols[e] == cols[k]:
            e += 1
        out.append(f"{e - k}{cols[k]}")
        k = e
    return "".join(out)


def replay(x, y, cigar, db_start, q_start, igap, egap):
    """walk the CIGAR over the reads: (score, db_end, q_end, matches, mismatches, gap columns, record length,
    record identities) with the record's counting rule (no start column, no match right after a gap run)"""
    score, i, j, mt, mm, gaps, cols, ids = 0, db_start, q_start, 0, 0, 0, 0, 0
    first, after_gap = True, False
    for n, op in CIGAR_RE.findall(cigar):
        n = int(n)
        if op in "ID":
            score += igap + n * egap
            gaps += n
            cols += n
            after_gap = True
            if op == "I":
                j += n
            else:
                i += n
            continue
        for _ in range(n):
            eq = x[i] == y[j]
            assert eq == (op == "="), (cigar, i, j)
            score += 4 if eq else -4
            mt += eq
            mm += not eq
            ids += eq and not first and not after_gap
            first = after_gap = False
            i += 1
            j += 1
            cols += 1
    return score, i, j, mt, mm, gaps, cols - 1, ids


def read(seq, start, k):
    return bytes(seq[int(start[k]):int(start[k + 1])])


def check_records(best, aln, off, ops, db, query, igap=-5, egap=-2):
    """every accepted record: replay == reported score / counts / coordinates / length / identities; others empty"""
    from imsame_b200 import api
    nq = len(query[1]) - 1
    n = 0
    for k, b in enumerate(best):
        a, c = aln[k], api.cigar_string(ops[int(off[k]):int(off[k + 1])])
        if not b["accepted"]:
            assert c == "" and not any(int(a[f]) for f in api.ALN_DTYPE.names)
            continue
        x, y = read(db[0], db[1], int(b["db_seq"])), read(query[0], query[1], k % nq)
        s, de, qe, mt, mm, gaps, ln, ids = replay(x, y, c, int(a["db_start"]), int(a["q_start"]), igap, egap)
        assert (s, de, qe, mt, mm, gaps) == (int(a["score"]), int(a["db_end"]), int(a["q_end"]), int(a["matches"]),
                                              int(a["mismatches"]), int(a["gap_cols"])), (k, c)
        assert min(int(a["db_start"]), int(a["q_start"])) == 0 and a["db_end"] <= len(x) and a["q_end"] <= len(y)
        assert (ln, ids) == (int(b["length"]), int(b["identities"])), (k, c)
        # identity and coverage as the record line prints them
        assert api.header_fields(k % nq, {"length": ln, "identities": ids, "db_seq": b["db_seq"]}, len(y)) == \
            api.header_fields(k % nq, b, len(y))
        n += 1
    return n


def pair_records(gpu, xs, ys, igap, egap):
    """explicit pairs as a database and a query of the same size, record r = pair r with the forward NW's length and
    identities (imsame_gpu_nw_batch): every pair gets traced, accepted by a filter or not"""
    from imsame_b200 import api
    nw, _ = gpu.nw_batch(xs, ys, igap=igap, egap=egap)  # given positive, like make_params
    cat = lambda rs: (np.concatenate(rs).astype(np.uint8), np.concatenate([[0], np.cumsum([len(r) for r in rs])]).astype(np.uint64))
    best = np.zeros(len(xs), dtype=api.BEST_DTYPE)
    best["db_seq"] = np.arange(len(xs))
    best["length"], best["identities"], best["accepted"] = nw[:, 3], nw[:, 4], 1
    return cat(xs), cat(ys), best, nw


# ---- CPU -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("args", [["600", "3"], ["150", "9", "2999"]])  # reads of up to 3000 bases: 12 passes
def test_cigar_device_functions_on_cpu(args, tmp_path):
    """cigar.cuh's wavefront with 4-bit codes + walk, stepped as a warp on the CPU: the forward NW of the oracle, the
    winners' 16-bit path op for op, and the replay of every CIGAR"""
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    o = str(tmp_path / "orc.o")
    subprocess.check_call([cc, "-O2", "-c", os.path.join(hp.ROOT, "oracle", "imsame_oracle.c"), "-o", o])
    exe = str(tmp_path / "cigar_emul")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(hp.ROOT, "tests", "emul", "cigar_emul.cpp"),
                           o, "-lm"])
    r = subprocess.run([exe] + args, capture_output=True, text=True)
    assert r.returncode == 0 and "0 mismatches" in r.stdout, r.stdout[-2000:]


def test_reference_dp_matches_the_oracle(built):
    """the Python reference gives the oracle's forward NW (score, best cell, length, identities by the record rule)"""
    lib, u8p = hp.oracle(), C.POINTER(C.c_ubyte)
    xs, ys = sc.random_pairs(31, 60, max_len=120)
    for k, (x, y) in enumerate(zip(xs, ys)):
        if len(x) < 2 or len(y) < 2:
            continue
        igap, egap = [(-5, -2), (-3, -1), (0, 0), (2, 1)][k % 4]
        s, bx, by, cig, (x0, y0) = ref_nw(bytes(x), bytes(y), igap, egap)
        o = [C.c_int32(), C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()]
        lib.orc_nw_forward(x.ctypes.data_as(u8p), len(x), y.ctypes.data_as(u8p), len(y), igap, egap, *[C.byref(v) for v in o])
        rs, de, qe, mt, mm, gaps, ln, ids = replay(bytes(x), bytes(y), cig, x0, y0, igap, egap)
        assert (s, bx, by, ln, ids) == tuple(v.value for v in o) and (rs, de, qe) == (s, bx + 1, by + 1), k


def test_cigar_string():
    from imsame_b200 import api
    ops = [5 << 4 | 7, 1 << 4 | 8, 2 << 4 | 2, 3 << 4 | 7, 4 << 4 | 1, 1 << 4 | 7]
    assert api.cigar_string(ops) == "5=1X2D3=4I1="
    assert api.cigar_string(ops, extended=False) == "6M2D3M4I1M"
    assert api.cigar_string([]) == ""


# ---- GPU -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("gaps", [(5, 2), (3, 1), (0, 0)])
def test_random_pairs_against_the_reference_dp(gpu, gaps):
    """a few hundred pairs (noisy copies with indels, random pairs, tiny reads): score, best cell and CIGAR identical to
    the Python reference; the replay of every CIGAR gives the reported numbers"""
    from imsame_b200 import api
    xs, ys = sc.random_pairs(100 + gaps[0], 240, max_len=160)
    xs, ys = zip(*[(x, y) for x, y in zip(xs, ys) if len(x) >= 2 and len(y) >= 2])
    db, q, best, nw = pair_records(gpu, xs, ys, *gaps)
    p = api.make_params(igap=gaps[0], egap=gaps[1])
    aln, off, ops = gpu.align_traceback(db, q, best, p)
    assert check_records(best, aln, off, ops, db, q, -gaps[0], -gaps[1]) == len(xs)
    for k, (x, y) in enumerate(zip(xs, ys)):
        s, bx, by, cig, (x0, y0) = ref_nw(bytes(x), bytes(y), -gaps[0], -gaps[1])
        assert s == int(aln[k]["score"]) == int(nw[k, 0]) and (bx, by) == (int(nw[k, 1]), int(nw[k, 2]))
        assert api.cigar_string(ops[int(off[k]):int(off[k + 1])]) == cig, k
        assert (int(aln[k]["db_start"]), int(aln[k]["q_start"]), int(aln[k]["db_end"]), int(aln[k]["q_end"])) == (x0, y0, bx + 1, by + 1)


@pytest.mark.gpu
def test_edge_cases(gpu):
    """identical reads (one '=' run over both reads, touching all four ends), the smallest pairs, alignments that are
    almost all gap on either side, reads of almost 3000 bases"""
    from imsame_b200 import api
    rng = np.random.default_rng(5)
    B = np.frombuffer(b"ACGT", dtype=np.uint8)
    r = lambda n: np.ascontiguousarray(B[rng.integers(0, 4, size=n)])
    a, b, c, long_ = r(300), r(300), r(2), r(2950)  # 2950 + 40 inserted bases: within the 3000-base limit
    xs = [a, c, a, np.concatenate([b[:20], b[-20:]]), r(2), long_, long_]
    ys = [a.copy(), c.copy(), np.concatenate([a[:20], a[-20:]]), b, r(7), long_.copy(), np.concatenate([long_[:1500], r(40), long_[1500:]])]
    db, q, best, nw = pair_records(gpu, xs, ys, 0, 0)
    aln, off, ops = gpu.align_traceback(db, q, best, api.make_params(igap=0, egap=0))
    assert check_records(best, aln, off, ops, db, q, 0, 0) == len(xs)
    cig = [api.cigar_string(ops[int(off[k]):int(off[k + 1])]) for k in range(len(xs))]
    assert cig[0] == "300=" and cig[5] == "2950="
    assert tuple(int(aln[0][f]) for f in ("q_start", "q_end", "db_start", "db_end")) == (0, 300, 0, 300)
    assert int(aln[2]["gap_cols"]) > 0 and int(aln[3]["gap_cols"]) > 0
    assert "I" in cig[6]
    for k, (x, y) in enumerate(zip(xs, ys)):
        if len(x) * len(y) < 200000:
            assert ref_nw(bytes(x), bytes(y), 0, 0)[3] == cig[k], k
    # rewarded gaps (igap = egap = +2 as stored): paths of almost nothing but gap runs, on either side
    xs, ys = [a, np.concatenate([b[:20], b[-20:]])], [np.concatenate([a[:20], a[-20:]]), b]
    db, q, best, nw = pair_records(gpu, xs, ys, -2, -2)
    aln, off, ops = gpu.align_traceback(db, q, best, api.make_params(igap=-2, egap=-2))
    assert check_records(best, aln, off, ops, db, q, 2, 2) == 2
    for k, (x, y) in enumerate(zip(xs, ys)):
        assert int(aln[k]["gap_cols"]) > int(aln[k]["matches"]) + int(aln[k]["mismatches"])
        assert ref_nw(bytes(x), bytes(y), 2, 2)[3] == api.cigar_string(ops[int(off[k]):int(off[k + 1])]), k


@pytest.mark.gpu
def test_zero_accepted_records(gpu):
    from imsame_b200 import api
    db, ds, q, qs = sc.fixed_case(7, 2, 20000, 150, 300, 50, 0.03)
    best = np.zeros(50, dtype=api.BEST_DTYPE)
    aln, off, ops = gpu.align_traceback((db, ds), (q, qs), best)
    assert len(ops) == 0 and not off.any() and not aln.view(np.uint32).any()


@pytest.fixture(scope="module")
def whole_run(gpu):
    """a whole-path run on ragged reads (fixed-length runs are the golden tests below)"""
    from imsame_b200 import api
    db, ds, q, qs = sc.ragged_case(41, 3, 40000, 3000, 600, 0.05, lo=40, hi=320)
    out, _ = gpu.align((db, ds), (q, qs), api.make_params())
    assert out["accepted"].sum() > 100
    return (db, ds), (q, qs), out


@pytest.mark.gpu
def test_whole_path_records_replay(gpu, whole_run):
    d, q, out = whole_run
    aln, off, ops = gpu.align_traceback(d, q, out)
    assert check_records(out, aln, off, ops, d, q) == out["accepted"].sum()


@pytest.mark.gpu
def test_a_small_budget_splits_the_batch_with_the_same_result(gpu, whole_run, monkeypatch):
    d, q, out = whole_run
    want = gpu.align_traceback(d, q, out)
    monkeypatch.setenv("IMSAME_TRACEBACK_BUDGET", "200000")  # a few hits per batch
    got = gpu.align_traceback(d, q, out)
    monkeypatch.setenv("IMSAME_TRACEBACK_BUDGET", "1")  # one hit per batch
    one = gpu.align_traceback(d, q, out)
    for w, g, o in zip(want, got, one):
        assert np.array_equal(w, g) and np.array_equal(w, o)


@pytest.mark.gpu
def test_records_of_another_database_are_an_error(gpu, whole_run):
    from imsame_b200 import api
    (db, ds), q, out = whole_run
    with pytest.raises(api.ImsameError) as e:
        gpu.align_traceback((COMP[db[::-1]].copy(), (len(db) - ds[::-1]).astype(np.uint64)), q, out)
    assert e.value.code == -3
    gpu.align_traceback((db, ds), q, out)  # the context stays usable


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["synth150", "dirty"])
def test_golden_inputs(gpu, name):
    from imsame_b200 import api, hostlib as H
    seq, start, brk = H.load_fasta(os.path.join(G, f"{name}.db.fa"), True)
    q, qs, _ = H.load_fasta(os.path.join(G, f"{name}.q.fa"), False)
    gaps = (4, 1) if name == "dirty" else (5, 2)
    p = api.make_params(min_coverage=0.3 if name == "dirty" else 0.5, min_identity=0.6 if name == "dirty" else 0.5,
                        min_e_value=1e-10 if name == "dirty" else None, igap=gaps[0], egap=gaps[1])
    out, _ = gpu.align((seq, start), (q, qs), p, db_breaks=brk)
    aln, off, ops = gpu.align_traceback((seq, start), (q, qs), out, p)
    assert check_records(out, aln, off, ops, (seq, start), (q, qs), -gaps[0], -gaps[1]) == out["accepted"].sum() > 10


@pytest.mark.gpu
def test_reverse_strand_records(gpu):
    """records of align_revcomp() are traced against the reverse complement database they index; the same as tracing
    the records of a run against that database directly"""
    from imsame_b200 import api
    db, ds, q, qs = sc.fixed_case(43, 3, 40000, 250, 3000, 500, 0.05)
    lens = np.diff(ds.astype(np.int64))
    db = db.copy()
    for i in range(1, len(lens), 2):  # reads of both strands
        s, e = int(ds[i]), int(ds[i + 1])
        db[s:e] = COMP[db[s:e][::-1]]
    rdb = (COMP[db[::-1]].copy(), (len(db) - ds[::-1].astype(np.int64)).astype(np.uint64))
    p = api.make_params()
    gpu.align((db, ds), (q, qs), p)
    rev, _ = gpu.align_revcomp()
    assert rev["accepted"].sum() > 50
    got = gpu.align_traceback(rdb, (q, qs), rev, p)
    assert check_records(rev, *got, rdb, (q, qs)) == rev["accepted"].sum()
    direct, _ = gpu.align(rdb, (q, qs), p)
    assert np.array_equal(direct, rev)
    for w, g in zip(gpu.align_traceback(rdb, (q, qs), direct, p), got):
        assert np.array_equal(w, g)


@pytest.mark.gpu
def test_sweep_sets(gpu, whole_run):
    """the sets of a sweep in one call: block t == the call on set t alone; pairs shared by sets are traced once"""
    from imsame_b200 import api
    d, q, _ = whole_run
    ps = [api.make_params(min_coverage=c, min_identity=i) for c, i in ((0.5, 0.5), (0.7, 0.8), (0.9, 0.95))]
    sets, codes, _ = gpu.align_sweep(d, q, ps)
    assert codes == [0, 0, 0]
    aln, off, ops = gpu.align_traceback(d, q, sets)
    nq = len(q[1]) - 1
    for t, s in enumerate(sets):
        a1, o1, p1 = gpu.align_traceback(d, q, s)
        assert np.array_equal(aln[t * nq:(t + 1) * nq], a1)
        for r in range(nq):
            k = t * nq + r
            assert np.array_equal(ops[int(off[k]):int(off[k + 1])], p1[int(o1[r]):int(o1[r + 1])])
        assert check_records(s, a1, o1, p1, d, q) == s["accepted"].sum() > 0


def strip_columns(text):
    return re.sub(rb"(?m)^(\(\d+, \d+\) : \d+% \d+% \d+)( .*)$", rb"\1", text)


def check_cigar_file(path, db, query, igap=-5, egap=-2):
    """every header line has the columns and they replay; returns the number of records"""
    n = 0
    for line in open(path, "rb").read().split(b"\n"):
        if not line.startswith(b"("):
            continue
        m = COLS_RE.match(line)
        assert m, line
        r, s, pi, pc, ylen, q0, q1, d0, d1, score = (int(v) for v in m.groups()[:10])
        x, y = read(db[0], db[1], s), read(query[0], query[1], r)
        got = replay(x, y, m.group(11).decode(), d0, q0, igap, egap)
        assert got[:3] == (score, d1, q1) and ylen == len(y), line
        ln, ids = got[6], got[7]
        assert (pi, pc) == (min(100, 100 * ids // ln), min(100, 100 * ln // ylen)), line
        n += 1
    return n


@pytest.mark.gpu
def test_cli_cigar_columns(gpu, tmp_path):
    """IMSAME without -cigar writes what it wrote before (the golden file); with -cigar every header line gains the
    columns, which replay over the reads; -out_rev and -sweep files too"""
    from imsame_b200 import hostlib as H
    qf, dbf = os.path.join(G, "synth150.q.fa"), os.path.join(G, "synth150.db.fa")
    plain, cig, rev, sw = (str(tmp_path / n) for n in ("plain.align", "cigar.align", "cigar.r.align", "sweep.align"))
    subprocess.check_call([EXE, "-query", qf, "-db", dbf, "-out", plain, "-n_threads", "1"], stdout=subprocess.DEVNULL)
    assert open(plain, "rb").read() == open(os.path.join(G, "synth150.t1.align"), "rb").read()
    subprocess.check_call([EXE, "-query", qf, "-db", dbf, "-out", cig, "-out_rev", rev, "-n_threads", "1", "-cigar"],
                          stdout=subprocess.DEVNULL)
    assert strip_columns(open(cig, "rb").read()) == open(plain, "rb").read()
    seq, start, _ = H.load_fasta(dbf, True)
    q, qs, _ = H.load_fasta(qf, False)
    assert check_cigar_file(cig, (seq, start), (q, qs)) > 10
    rf = str(tmp_path / "db.r.fa")
    subprocess.check_call([REVCOMP, dbf, rf], stdout=subprocess.DEVNULL)
    rseq, rstart, _ = H.load_fasta(rf, True)
    check_cigar_file(rev, (rseq, rstart), (q, qs))
    subprocess.check_call([EXE, "-query", qf, "-db", dbf, "-out", sw, "-n_threads", "1", "-cigar", "-sweep", "0.8:0.9"],
                          stdout=subprocess.DEVNULL)
    assert open(sw, "rb").read() == open(cig, "rb").read()
    assert check_cigar_file(sw + ".1", (seq, start), (q, qs)) > 0


@pytest.mark.gpu
def test_allvsall_cigar_jobs2_equals_jobs1(gpu, tmp_path):
    """IMSAME_allvsall -cigar: -jobs 2 writes the files of -jobs 1; without -cigar the files are those minus the
    columns; the columns replay (X-Y.r.align against the reverse complement sample)"""
    from imsame_b200 import hostlib as H
    d = tmp_path / "samples"
    d.mkdir()
    pool = H.SynthPool(4003, 3, 30000)
    for i in range(3):
        H.write_fasta(str(d / f"s{i}.fasta"), pool.db_reads(i * 700, 400, 150), 400, 150, "r")
    pool.close()
    outs = {}
    for tag, extra in (("j1", ["-cigar"]), ("j2", ["-cigar", "-jobs", "2"]), ("plain", [])):
        o = tmp_path / tag
        o.mkdir()
        r = subprocess.run([ALLVSALL, str(d), "0.5", "0.5", "4", "fasta", str(o)] + extra, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        outs[tag] = {n: open(o / n, "rb").read() for n in sorted(os.listdir(o))}
    assert outs["j1"] == outs["j2"] and len(outs["j1"]) == 6
    assert {n: strip_columns(t) for n, t in outs["j1"].items()} == outs["plain"]
    n = 0
    for name in outs["j1"]:
        m = re.match(r"s(\d)-s(\d)(\.r)?\.align$", name)
        qf, dbf = str(d / f"s{m.group(1)}.fasta"), str(d / f"s{m.group(2)}.fasta")
        if m.group(3):
            rf = str(tmp_path / "rev.fa")
            subprocess.check_call([REVCOMP, dbf, rf], stdout=subprocess.DEVNULL)
            dbf = rf
        seq, start, _ = H.load_fasta(dbf, True)
        q, qs, _ = H.load_fasta(qf, False)
        n += check_cigar_file(str(tmp_path / "j1" / name), (seq, start), (q, qs))
    assert n > 100
