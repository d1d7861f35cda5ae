"""GPU tests added in the last session of round 2 without a GPU at hand (named to run after the other GPU files).

1. All-vs-all on samples whose reverse complement is NOT the mirror image of the sample (GPU; named to run after the
other GPU files).  revComp keeps letters only (src/reverseComplement.c:65-70) while the database loader restarts the
seed word at every dropped character but the newline (src/IMSAME.c:229-231): in a multi-line CRLF file, or one with
gap characters inside its records, the sample has word breaks its reverse complement does not have; 'U' comes back
as an 'A' the loader keeps.  bin/IMSAME_allvsall may derive a reverse-complemented read set on the device only when
imsame_revcomp_is_mirror says so (tests/test_host_cpu.py pins that predicate on the CPU); here the outputs of the
in-process driver are compared with the script's (one IMSAME + revComp process per comparison, text all the way) and,
when oracle/_ref travelled, with the unmodified reference workflow.  The samples hold reverse-strand reads so that
the .r.align files are not empty.

2. The whole path and the winners' traceback on LONG reads (400..2900 bases): extension walks of up to ~90 windows
through the scan kernel's park queue, the generic NW kernel in up to 12 balanced passes, back-pointer tables of up
to 2900 x 3072 codes -- the other whole-path tests stop at 450 bases (the device functions themselves are covered
at these lengths by tests/emul on the CPU and by test_nw_batch_matches_oracle on the GPU)."""
import ctypes as C
import os
import subprocess

import numpy as np

import pytest

import helpers as hp
import synth_cases as sc

pytestmark = pytest.mark.gpu


def test_all_vs_all_with_samples_that_are_not_their_mirror(gpu, tmp_path):
    d, o1, o2, o3 = (tmp_path / n for n in ("samples", "out_script", "out_batch", "out_reference"))
    for p in (d, o1, o2, o3):
        p.mkdir()
    sc.write_allvsall_filter_samples(d)
    from imsame_b200 import hostlib as H
    assert not H.revcomp_is_mirror((d / "s1.fasta").read_bytes()) and not H.revcomp_is_mirror((d / "s2.fasta").read_bytes())
    assert H.revcomp_is_mirror((d / "s0.fasta").read_bytes()) and H.revcomp_is_mirror((d / "s3.fasta").read_bytes())
    args = [str(d), "0.5", "0.5", "2", "fasta"]
    subprocess.run([os.path.join(hp.ROOT, "bin", "all_vs_all_metagenomes_IMSAME.sh")] + args + [str(o1)],
                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    r = subprocess.run([os.path.join(hp.ROOT, "bin", "IMSAME_allvsall")] + args + [str(o2)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    names = sorted(os.listdir(o1))
    assert names == sorted(os.listdir(o2)) and len(names) == 12
    for n in names:
        assert open(o1 / n, "rb").read() == open(o2 / n, "rb").read(), n
    # the reverse-strand samples match the forward one through their reverse complement
    for n in ("s0-s1.r.align", "s0-s2.r.align", "s0-s3.r.align"):
        assert os.path.getsize(o2 / n) > 5000, n
    # the query-s0 files against what the reference workflow wrote (tests/golden/reference_pins.json)
    want = hp.pins("allvsall_text_filter_samples")
    for n in want:
        assert hp.align_digest(str(o2 / n), lines=True) == want[n], n
    ref_script = os.path.join(hp.ROOT, "oracle", "_ref", "all_vs_all_metagenomes_IMSAME.sh")
    if os.path.exists(ref_script) and hp.have_reference():
        subprocess.run(["bash", ref_script] + args + [str(o3)], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        assert sorted(os.listdir(o3)) == names
        for n in names:  # two threads share the reference's output stream: header sets and sorted lines (tools/allvsall_bench.py)
            assert hp.parse_align_headers(str(o3 / n)) == hp.parse_align_headers(str(o2 / n)), n
            assert sorted(open(o3 / n, "rb").read().split(b"\n")) == sorted(open(o2 / n, "rb").read().split(b"\n")), n


def test_long_reads_whole_path_and_traceback_match_the_oracle(gpu):
    from imsame_b200 import api, hostlib as H
    db, ds, q, qs = sc.ragged_case(6061, 2, 30000, 400, 90, 0.05, lo=400, hi=2900)
    odb, oq = hp.OracleSeqs(seq=db, start=ds), hp.OracleSeqs(seq=q, start=qs)
    best, _ = hp.oracle_align(odb, oq, hp.default_params(n_threads=3))
    want = hp.best_to_records(best, len(qs) - 1)
    assert len(want) > 30 and max(int(qs[r + 1] - qs[r]) for r in want) > 2500
    p = api.make_params(n_threads=3)
    out, _ = gpu.align((db, ds), (q, qs), p)
    got = {int(r): (int(o["db_seq"]), int(o["qpos_end"]), int(o["db_pos"]), int(o["length"]), int(o["identities"]))
           for r, o in enumerate(out) if o["accepted"]}
    assert got == want
    ops_off, ops, cell = gpu.traceback((db, ds), (q, qs), out, p)
    lib = hp.oracle()
    u8p = C.POINTER(C.c_ubyte)
    for r in sorted(want):
        s = int(out[r]["db_seq"])
        x = np.ascontiguousarray(db[int(ds[s]):int(ds[s + 1])])
        y = np.ascontiguousarray(q[int(qs[r]):int(qs[r + 1])])
        text = C.create_string_buffer(8 * (len(x) + len(y)) + 512)
        sc_, bx, by, ln, idn = C.c_int32(), C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
        lib.orc_nw_traceback(x.ctypes.data_as(u8p), len(x), y.ctypes.data_as(u8p), len(y), -5, -2, C.byref(sc_),
                             C.byref(bx), C.byref(by), C.byref(ln), C.byref(idn), text, len(text))
        rec = H.render_record(int(r), s, int(out[r]["length"]), int(out[r]["identities"]), x, y, cell[r, 0],
                              cell[r, 1], ops[int(ops_off[r]):int(ops_off[r + 1])])
        hdr_len = rec.index(b" $$$$$$$ \n") + len(b" $$$$$$$ \n")
        assert rec[hdr_len:] == text.value, r
        assert (int(cell[r, 0]), int(cell[r, 1]), int(out[r]["length"]), int(out[r]["identities"])) == \
            (bx.value, by.value, ln.value, idn.value)
