"""Host-side C (no GPU): FASTA ingest, exact threshold tables, renderer + device-function
emulators, revComp, C-ABI symbol export, CLI argument handling."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as hp
import synth_cases as sc

G = os.path.join(hp.ROOT, "tests", "golden")


@pytest.mark.parametrize("name,is_db", [("dirty.db.fa", True), ("dirty.q.fa", False), ("synth150.db.fa", True)])
def test_fasta_loader_matches_oracle_loader(built, name, is_db):
    from imsame_b200 import hostlib as H
    seq, start, brk = H.load_fasta(os.path.join(G, name), is_db)
    o = hp.OracleSeqs(os.path.join(G, name), is_db)
    oseq, ostart, obrk = o.numpy()
    assert np.array_equal(seq, oseq) and np.array_equal(start, ostart)
    if is_db:
        assert np.array_equal(brk, obrk)
        if name.startswith("dirty"):
            assert len(brk) > 10
    assert set(np.unique(seq)) <= set(b"ACGT")


@pytest.mark.parametrize("is_db", [True, False])
def test_parallel_fasta_loader_on_a_dirty_multi_megabyte_file(built, is_db, tmp_path):
    """the loader cuts files > 1 MB into pieces at "\\n>" and parses them on all threads: records that
    start mid-line, '>' inside headers, N runs, CRLF, lower case, empty records, text before the first
    header and a missing final newline must come out exactly as in the sequential oracle loader"""
    from imsame_b200 import hostlib as H
    rng = np.random.default_rng(5 + int(is_db))
    alpha = np.frombuffer(b"ACGTACGTACGTacgtNnRY-", dtype=np.uint8)
    parts = [b"junk before the first header\nACGT\n"]
    for r in range(9000):
        hdr = b">r%d desc > with gt" % r if r % 7 else b">r%d" % r
        parts.append(hdr + (b"\r\n" if r % 5 == 0 else b"\n"))
        if r % 97 == 0:
            continue  # empty record
        for _ in range(int(rng.integers(1, 9))):
            line = alpha[rng.integers(0, len(alpha), size=int(rng.integers(1, 120)))].tobytes()
            parts.append(line + (b"\r\n" if r % 5 == 0 else b"\n"))
        if r % 211 == 0:
            parts.append(b"ACGTAC>midline record start\nGGGTTTAAACCC")  # '>' not at a line start, no newline after
            parts.append(b"\n")
    parts.append(b">last\nACGTNACGT")  # no final newline
    path = str(tmp_path / "big_dirty.fa")
    open(path, "wb").write(b"".join(parts))
    assert os.path.getsize(path) > 2 * (1 << 20)
    seq, start, brk = H.load_fasta(path, is_db)
    o = hp.OracleSeqs(path, is_db)
    oseq, ostart, obrk = o.numpy()
    assert np.array_equal(start, ostart)
    assert np.array_equal(seq, oseq)
    if is_db:
        assert np.array_equal(brk, obrk) and len(brk) > 1000


def test_threshold_tables_are_exact(built):
    from imsame_b200 import api, hostlib as H
    lib = hp.oracle()
    for min_e, total in ((api.default_evalue(), 15_000_000), (1e-5, 2_500_000_000), (0.5, 1000)):
        nmin, lmin, imin = H.threshold_tables(min_e, 0.5, 0.5, total)
        for ylen in (11, 12, 100, 150, 250, 2999, 3000):
            n = int(nmin[ylen])
            if n == 65535:
                continue
            assert lib.orc_evalue(n, ylen, total) < min_e
            if n > 0:
                assert not (lib.orc_evalue(n - 1, ylen, total) < min_e)
    assert int(H.threshold_tables(api.default_evalue(), 0.5, 0.5, 15_000_000)[0][150]) == 61  # SURVEY 8(a) A3
    assert int(H.threshold_tables(api.default_evalue(), 0.5, 0.5, 2_500_000_000)[0][250]) == 66
    for cov, ident in ((0.5, 0.5), (0.3, 0.6), (0.8, 0.9), (1.0, 1.0)):
        _, lmin, imin = H.threshold_tables(1e-20, cov, ident, 1000)
        ld = np.longdouble
        for ylen in (1, 7, 150, 250, 3000):
            l = int(lmin[ylen])
            assert ld(l) / ld(ylen) >= ld(cov) and not (ld(l - 1) / ld(ylen) >= ld(cov))
        for ln in (1, 10, 149, 300, 6000):
            i = int(imin[ln])
            assert ld(i) / ld(ln) >= ld(ident) and (i == 0 or not (ld(i - 1) / ld(ln) >= ld(ident)))
        assert imin[0] == 65535


@pytest.mark.parametrize("prog,args", [("nw_emul", ["400", "3"]), ("nwp_emul", ["3000", "5"]), ("extend_emul", ["5"]),
                                       ("extend_emul", ["6", "8"]), ("extend_emul", ["7", "15"]),
                                       ("extend_emul", ["5", "12", "3000"]),  # reads of up to 3000 bases: walks of ~100 windows
                                       ("tb_emul", ["300", "4"]), ("tb_emul", ["400", "9", "2989"])])  # reads of up to 3000 bases
def test_device_functions_on_cpu(built, prog, args, tmp_path):
    """the HD functions the kernels are made of (nw_core.cuh, nwp_core.cuh, extend.cuh, traceback.cuh) + render.c,
    compiled for the host and stepped as a 32-lane warp, against the oracle"""
    exe = str(tmp_path / prog)
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    objs = []
    for src in ("oracle/imsame_oracle.c", "imsame_b200/host/render.c"):
        o = str(tmp_path / (os.path.basename(src) + ".o"))
        subprocess.check_call([cc, "-O2", "-c", os.path.join(hp.ROOT, src), "-o", o])
        objs.append(o)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(hp.ROOT, "tests", "emul", prog + ".cpp")]
                          + objs + ["-lm"])
    r = subprocess.run([exe] + args, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:]
    assert "0 mismatches" in r.stdout


def test_revcomp_matches_reference_semantics(built, tmp_path):
    src = tmp_path / "in.fa"
    src.write_bytes(b">a x\nACGTNnacgu\nGG\n>b\nTTTT\nCA\n>c only header\n>d\nacgtRYKM\n")
    out = tmp_path / "out.fa"
    subprocess.check_call([os.path.join(hp.ROOT, "bin", "revComp"), str(src), str(out)])
    assert out.read_bytes() == b">d\nMKYRacgt\n>c only header\n\n>b\nTGAAAA\n>a x\nCCacgtnNACGT\n"
    out2 = tmp_path / "out2.fa"
    subprocess.check_call([os.path.join(hp.ROOT, "bin", "revComp"), os.path.join(G, "dirty.db.fa"), str(out2)])
    assert hp.sha(out2.read_bytes()) == hp.pins("revcomp_dirty_db")
    if os.path.exists(hp.REF_REVCOMP):
        ref = tmp_path / "ref.fa"
        subprocess.check_call([hp.REF_REVCOMP, str(src), str(ref)])
        assert ref.read_bytes() == out.read_bytes()
        ref2 = tmp_path / "ref2.fa"
        subprocess.check_call([hp.REF_REVCOMP, os.path.join(G, "dirty.db.fa"), str(ref2)])
        assert ref2.read_bytes() == out2.read_bytes()


def test_revcomp_header_lines_with_many_record_starts(built, tmp_path):
    """every '>' byte starts a record (src/reverseComplement.c:47-52) and a record's header runs to the end of its
    line (:59), so a line holding m '>' bytes comes out m times: the output is longer than twice the input (the
    first implementation sized its buffer 2 n + 16 and overflowed; found by fuzzing against the reference tool)"""
    src = tmp_path / "in.fa"
    line = b">" * 40 + b"tail of the line" * 4 + b"\n"
    src.write_bytes(b">first rec\nACGT\n" + line + b"ACGTTGCA\n" + line)
    out = tmp_path / "out.fa"
    subprocess.check_call([os.path.join(hp.ROOT, "bin", "revComp"), str(src), str(out)])
    got = out.read_bytes()
    assert len(got) > 2 * len(src.read_bytes()) + 16
    want = b""
    for body in (b"", b"TGCAACGT"):  # records in reverse file order; all 40 of a line share the body after it
        for k in range(40):  # the last '>' of the line first
            want += b">" * (k + 1) + b"tail of the line" * 4 + b"\n" + body + b"\n"
    want += b">first rec\nACGT\n"
    assert got == want
    if os.path.exists(hp.REF_REVCOMP):
        ref = tmp_path / "ref.fa"
        subprocess.check_call([hp.REF_REVCOMP, str(src), str(ref)])
        assert ref.read_bytes() == got


def test_revcomp_fuzz_against_the_reference_tool(built, tmp_path):
    """seeded random byte soup (record starts anywhere, CRLF, tabs, U/u, IUPAC letters, empty files): same output
    file, same stdout, same exit status as the compiled reference tool where oracle/_ref is built; what it gave is
    pinned in tests/golden/reference_pins.json"""
    got = revcomp_fuzz(str(tmp_path), os.path.exists(hp.REF_REVCOMP))
    assert got == hp.pins("revcomp_fuzz")


def revcomp_fuzz(d, live):
    """bin/revComp on the seeded cases, compared with the reference tool when `live`: per case (exit status, stdout,
    output file) as digests"""
    rng = np.random.default_rng(5)
    tokens = [b"A", b"C", b"G", b"T", b"a", b"c", b"g", b"t", b"N", b"n", b"\n", b"\r\n", b">", b">h\n", b" ", b"-", b"U", b"u",
              b"R", b"\t", b"ACGTACGTACGTACGTACGTTTGGCCAA", b"\n>x y\n", b"\n\n", b">\n"]
    src, o1, o2 = (os.path.join(d, n) for n in ("in.fa", "o1", "o2"))
    compared, out = 0, []
    for it in range(400):
        body = b"".join(tokens[i] for i in rng.integers(0, len(tokens), size=int(rng.integers(0, 120))))
        if it % 2 == 0:
            body = b">first rec\n" + body
        open(src, "wb").write(body)
        for f_ in (o1, o2):
            if os.path.exists(f_):
                os.remove(f_)
        # every third case with the file cut into pieces of a few bytes (the threaded path of imsame_revcomp_mem)
        env = dict(os.environ, IMSAME_TEST_FASTA_PIECE=str(1 + it % 7)) if it % 3 == 0 else None
        r1 = subprocess.run([os.path.join(hp.ROOT, "bin", "revComp"), src, o1], capture_output=True, env=env)
        out.append([r1.returncode, hp.sha(r1.stdout), hp.sha(open(o1, "rb").read()) if os.path.exists(o1) else None])
        if live:
            r2 = subprocess.run([hp.REF_REVCOMP, src, o2], capture_output=True)
            if r2.returncode < 0:
                continue  # the reference itself died on a signal: nothing to compare with
            assert (r1.returncode, r1.stdout) == (r2.returncode, r2.stdout), (it, body)
            assert open(o1, "rb").read() == open(o2, "rb").read(), (it, body)
            compared += 1
    assert compared > 300 or not live
    return out


def test_device_revcomp_only_for_samples_whose_revcomp_is_their_mirror(built):
    """bin/IMSAME_allvsall derives the reverse-complemented read set on the device from the packed forward one only
    when revComp's text parses into exactly its mirror image (imsame_revcomp_is_mirror).  revComp keeps letters only
    (src/reverseComplement.c:65-70) while the database loader restarts the seed word at every dropped character but
    the newline (src/IMSAME.c:229-231): a CRLF file, gap characters, 'U' and repeated '>' all break the symmetry."""
    from imsame_b200 import hostlib as H
    body = b"ACGTTGCAGGCATTACGGATCCATGCAAGT"
    assert H.revcomp_is_mirror(b">a\n" + body + b"\n>b\n" + body[::-1] + b"\n" + body[:11] + b"\n>c x\nacgtacgtTTGA\n")
    assert H.revcomp_is_mirror(b">a\n" + body + b"N" + body + b"\n>b\nNN" + body + b"NN\n")  # letters break words both ways
    assert H.revcomp_is_mirror(b">only header\n")
    assert H.revcomp_is_mirror(b"")
    # multi-line records with CRLF: '\r' restarts the word in the sample, revComp drops it and writes one line
    assert not H.revcomp_is_mirror(b">a\r\n" + body + b"\r\n" + body + b"\r\n>b\r\n" + body + b"\r\n")
    assert H.revcomp_is_mirror(b">a\r\n" + body + b"\r\n>b\r\n" + body + b"\r\n")  # a trailing '\r' is no word break
    assert not H.revcomp_is_mirror(b">a\n" + body + b"-" + body + b"\n")      # gap character
    assert not H.revcomp_is_mirror(b">a\n" + body + b"*7 " + body + b"\n")
    assert not H.revcomp_is_mirror(b">a\n" + body + b"U" + body + b"\n")      # U -> A, which the loader keeps
    assert not H.revcomp_is_mirror(b">a>b\n" + body + b"\n")                  # one record per '>' byte
    rng = np.random.default_rng(3)
    alphabet = np.frombuffer(b"ACGTacgtN", dtype=np.uint8)
    clean = b"".join(b">r%d\n" % i + alphabet[rng.choice(9, size=int(rng.integers(1, 300)), p=[.12] * 8 + [.04])].tobytes() + b"\n"
                     for i in range(500))
    assert H.revcomp_is_mirror(clean)
    assert not H.revcomp_is_mirror(clean + b">z\nAC-GT\n")


def test_allvsall_text_filter_samples_reference_workflow_vs_oracle(built, tmp_path):
    """The CPU half of tests/test_gpu_zz_allvsall_text_filters.py: on its four samples (multi-line CRLF, gap characters,
    'U', 'N') the UNMODIFIED reference workflow (oracle/_ref script + binaries) and the oracle fed with bin/revComp's
    text give the same records -- and aligning against the MIRROR of the forward parse (what a device-side reverse
    complement of the packed sample would be) does not, exactly for the samples imsame_revcomp_is_mirror rejects.
    Where oracle/_ref is not built, the reference workflow's files are represented by their digests in
    tests/golden/reference_pins.json."""
    from imsame_b200 import hostlib as H
    d, o3 = tmp_path / "samples", tmp_path / "out_reference"
    d.mkdir(); o3.mkdir()
    sc.write_allvsall_filter_samples(d)
    args = [str(d), "0.5", "0.5", "2", "fasta"]
    live = hp.have_reference()
    if live:
        subprocess.run(["bash", os.path.join(hp.ROOT, "oracle", "_ref", "all_vs_all_metagenomes_IMSAME.sh")] + args + [str(o3)],
                       stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        assert len(os.listdir(o3)) == 12
    p = hp.default_params(n_threads=2, coverage=0.5, identity=0.5)
    comp = np.zeros(256, dtype=np.uint8)
    for a, b in zip(b"ACGT", b"TGCA"):
        comp[a] = b
    for y, mirror_ok in (("s1", False), ("s2", False), ("s3", True)):
        text = (d / f"{y}.fasta").read_bytes()
        assert H.revcomp_is_mirror(text) == mirror_ok
        q = hp.OracleSeqs(str(d / "s0.fasta"), False)
        nq = int(q.s.n_seqs)
        for rev in (0, 1):
            dbf = str(d / f"{y}.fasta")
            if rev:
                dbf = str(tmp_path / f"{y}.r.fasta")
                subprocess.check_call([os.path.join(hp.ROOT, "bin", "revComp"), str(d / f"{y}.fasta"), dbf], stdout=subprocess.DEVNULL)
            oo, name = str(tmp_path / "orc.align"), f"s0-{y}{'.r' if rev else ''}.align"
            best, _ = hp.oracle_align(hp.OracleSeqs(dbf, True), q, p, out_path=oo)
            if live:
                assert hp.parse_align_headers(str(o3 / name)) == hp.parse_align_headers(oo), name
                assert sorted(open(o3 / name, "rb").read().split(b"\n")) == sorted(open(oo, "rb").read().split(b"\n")), name
            got = hp.align_digest(oo, lines=True)
            assert got == hp.pins("allvsall_text_filter_samples")[name], name
            if rev:
                assert got["records"] > 100 and os.path.getsize(oo) > 5000  # reverse-strand samples: records in the .r files
                fwd = hp.OracleSeqs(str(d / f"{y}.fasta"), True)  # owns the arrays numpy() views
                seq, start, brk = fwd.numpy()
                total = len(seq)
                mirror = hp.OracleSeqs(seq=comp[seq[::-1]].copy(), start=(total - start.astype(np.int64)[::-1]).astype(np.uint64),
                                       brk=np.sort(total - brk.astype(np.int64)).astype(np.uint64))
                b2, _ = hp.oracle_align(mirror, q, p)
                assert (hp.best_to_records(best, nq) == hp.best_to_records(b2, nq)) == mirror_ok, name


def test_host_fuzz_under_sanitizers(tmp_path):
    """tools/host_fuzz.c built with AddressSanitizer + UBSan: the threaded FASTA parser cut into pieces of a few
    bytes against a char-at-a-time model of the reference loader (src/IMSAME.c:193-285, :323-347), revComp and the
    parse of its output, the renderer on random paths with the buffer imsame_host.h promises"""
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    probe = tmp_path / "p.c"
    probe.write_text("int main(void){return 0;}")
    san = ["-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-fno-omit-frame-pointer"]
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0", OMP_NUM_THREADS="4")  # (LeakSanitizer refuses to run under ptrace)
    env.pop("LD_PRELOAD", None)
    if subprocess.run([cc, *san, str(probe), "-o", str(tmp_path / "p")], capture_output=True).returncode != 0 or \
            subprocess.run([str(tmp_path / "p")], capture_output=True, env=env).returncode != 0:
        pytest.skip("no usable sanitizer runtime here (gcc without libasan, or a kernel whose address-space layout it rejects)")
    omp = ["-fopenmp"] if subprocess.run([cc, "-fopenmp", str(probe), "-o", str(tmp_path / "p")], capture_output=True).returncode == 0 else []
    exe = str(tmp_path / "host_fuzz")
    host = os.path.join(hp.ROOT, "imsame_b200", "host")
    subprocess.check_call([cc, "-O1", "-g", "-Wall", *omp, *san, "-D_FILE_OFFSET_BITS=64", os.path.join(hp.ROOT, "tools", "host_fuzz.c"),
                           os.path.join(host, "fasta.c"), os.path.join(host, "render.c"), "-lm", "-o", exe])
    r = subprocess.run([exe, "500", "7"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "0 mismatches" in r.stdout and "2000 parses" in r.stdout


def test_c_abi_exports_every_declared_symbol(built):
    from imsame_b200 import api
    hdr = open(os.path.join(hp.ROOT, "include", "imsame_gpu.h")).read()
    declared = set(re.findall(r"\b(imsame_gpu_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(api.SYMBOLS), declared ^ set(api.SYMBOLS)
    lib = C.CDLL(api.GPU_SO)
    for name in sorted(declared):
        assert getattr(lib, name) is not None
    lib.imsame_gpu_strerror.restype = C.c_char_p
    assert lib.imsame_gpu_strerror(-5) == b"Read size reached for gapped alignment."


def test_no_gpu_means_error_not_fallback(built):
    """without a CUDA device the product path must fail loudly"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from imsame_b200 import api
    with pytest.raises(api.ImsameError) as e:
        api.Imsame(0)
    assert e.value.code == -1


def test_command_lines_fail_loudly_without_a_gpu(built, tmp_path):
    """no CPU fallback behind the command lines either: without an sm_100 device bin/IMSAME and bin/IMSAME_allvsall
    end with the reference's error form (terror: message on stdout, exit status 255) and write no record"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    d, o = tmp_path / "s", tmp_path / "o"
    d.mkdir(); o.mkdir()
    (d / "a.fasta").write_bytes(open(os.path.join(G, "dirty.q.fa"), "rb").read())
    (d / "b.fasta").write_bytes(open(os.path.join(G, "dirty.db.fa"), "rb").read())
    r = subprocess.run([os.path.join(hp.ROOT, "bin", "IMSAME"), "-query", str(d / "a.fasta"), "-db", str(d / "b.fasta"), "-out",
                        str(o / "x.align")], capture_output=True, text=True)
    assert r.returncode == 255 and "ERR**** GPU hot path failed: no usable sm_100 CUDA device" in r.stdout
    assert "from the query were found" not in r.stdout and os.path.getsize(o / "x.align") == 0
    r = subprocess.run([os.path.join(hp.ROOT, "bin", "IMSAME_allvsall"), str(d), "0.5", "0.5", "2", "fasta", str(o)],
                       capture_output=True, text=True)
    assert r.returncode == 255 and "ERR**** no usable GPU" in r.stdout
    assert not [n for n in os.listdir(o) if n != "x.align"]


def test_cli_flags_and_errors(built, tmp_path):
    exe = os.path.join(hp.ROOT, "bin", "IMSAME")
    r = subprocess.run([exe, "--help"], capture_output=True, text=True)
    assert r.returncode == 1 and "USAGE:" in r.stdout and "-n_threads" in r.stdout
    r = subprocess.run([exe, "-query", str(tmp_path / "missing.fa")], capture_output=True, text=True)
    assert r.returncode == 255 and r.stdout == "ERR**** A query and database is required ****\n"
    q = os.path.join(G, "dirty.q.fa")
    r = subprocess.run([exe, "-query", q, "-db", q, "-coverage", "0"], capture_output=True, text=True)
    assert r.returncode == 255 and "Min-coverage must be larger than zero" in r.stdout
    r = subprocess.run([exe, "-query", q, "-db", q, "-kmer", "17"], capture_output=True, text=True)
    assert r.returncode == 255 and "The seed length must be between 4 and 16" in r.stdout
    for i, args in enumerate((["--help"], ["-query", "nope"], ["-query", q, "-db", q, "-identity", "-1"])):
        a = subprocess.run([exe] + args, capture_output=True, text=True)
        assert [a.returncode, hp.sha(a.stdout.encode())] == hp.pins("cli_error_forms")[i], args
        if hp.have_reference():
            b = subprocess.run([hp.REF_BIN] + args, capture_output=True, text=True)
            assert (a.returncode, a.stdout) == (b.returncode, b.stdout)
