"""Seeded fuzz of the oracle against the UNMODIFIED reference binary (oracle/_ref/IMSAME, compiled by
oracle/build_ref.sh): ragged reads of 12..450 bases incl. reads shorter than a word's reach, dirty FASTA
(text before the first header, '>' inside headers, CRLF, lower case, N runs and other IUPAC letters, blanks,
multi-line records, missing final newline), indels, absent reads, and random flags (-n_threads 1..100 incl. more
threads than reads, -evalue, -coverage, -identity, -igap, -egap incl. 0).  With -n_threads 1 the .align files
must be byte-identical, otherwise the header sets; the accepted count of the summary line always.
780 further cases of the same generator were run while writing this test (0 differences; the reference
needs about 4 s per case for its tables, hence the small number here)."""
import os
import subprocess

import numpy as np
import pytest

import helpers as hp

B = np.frombuffer(b"ACGT", dtype=np.uint8)


@pytest.mark.parametrize("seed0", [11, 12])
def test_oracle_fuzz_vs_live_reference(seed0, tmp_path):
    got = fuzz_cases(seed0, str(tmp_path), hp.have_reference())
    assert got == hp.pins("oracle_fuzz")[str(seed0)]
    assert sum(c["records"] > 0 for c in got) >= len(got) // 3


def fuzz_cases(seed0, d, live):
    """the oracle on the seeded cases of seed0, compared with the reference binary when `live`; returns per case what
    the comparison looks at (pinned in tests/golden/reference_pins.json)"""
    out = []
    for case in range(5):
        rng = np.random.default_rng(seed0 * 100003 + case)
        G = int(rng.integers(1, 4)); Lg = int(rng.integers(300, 4000))
        genomes = [B[rng.integers(0, 4, size=Lg)] for _ in range(G)]
        def read(lo, hi, div, absent_p):
            L = int(rng.integers(lo, hi))
            if rng.random() < absent_p:
                return B[rng.integers(0, 4, size=L)].copy()
            g = genomes[int(rng.integers(0, G))]
            L = min(L, len(g))
            at = int(rng.integers(0, len(g) - L + 1))
            r = g[at:at + L].copy()
            m = rng.random(L) < div
            r[m] = B[rng.integers(0, 4, size=int(m.sum()))]
            # a few indels
            if rng.random() < 0.3 and L > 30:
                k = int(rng.integers(5, L - 5)); r = np.delete(r, slice(k, k + int(rng.integers(1, 4))))
            if rng.random() < 0.3 and L > 30:
                k = int(rng.integers(5, len(r) - 5)); r = np.insert(r, k, B[rng.integers(0, 4, size=int(rng.integers(1, 4)))])
            return r
        def fasta(path, reads, dirty):
            with open(path, "wb") as f:
                if dirty and rng.random() < 0.3: f.write(b"text before any header\nACGTAC\n")
                for i, r in enumerate(reads):
                    f.write(b">r%d some desc\n" % i if not (dirty and rng.random() < 0.1) else b">r%d > inner gt\r\n" % i)
                    s = r.tobytes()
                    if dirty:
                        s = bytearray(s)
                        for _ in range(int(rng.integers(0, 4))):
                            if len(s) > 2:
                                k = int(rng.integers(0, len(s)))
                                s[k:k] = [b"N", b"n", b"NNNN", b"R", b"-", b" ", b"\r"][int(rng.integers(0, 7))]
                        if rng.random() < 0.3: s = bytes(s).lower()
                        s = bytes(s)
                        w = int(rng.integers(20, 90)); s = b"\n".join(s[i:i + w] for i in range(0, len(s), w))
                    f.write(s + (b"\n" if not (dirty and i == len(reads) - 1 and rng.random() < 0.5) else b""))
        nd = int(rng.integers(5, 400)); nq = int(rng.integers(1, 80))
        lo = int(rng.choice([12, 13, 20, 60, 150])); hi = lo + int(rng.integers(1, 300))
        div = float(rng.choice([0.0, 0.02, 0.05, 0.1, 0.2]))
        dirty = rng.random() < 0.6
        dbr = [read(lo, hi, 0.005, 0.05) for _ in range(nd)]
        qr = [read(lo, hi, div, 0.3) for _ in range(nq)]
        dbf, qf, ro, oo = (os.path.join(d, n) for n in ("db.fa", "q.fa", "ref.align", "orc.align"))
        fasta(dbf, dbr, dirty); fasta(qf, qr, dirty)
        nt = int(rng.choice([1, 1, 2, 3, 4, 7, 8, 100]))
        ev = rng.choice([None, 1e-20, 1e-10, 1e-5, 1e-2, 0.5]); cov = float(rng.choice([0.5, 0.2, 0.8, 1.0, 0.01])); idn = float(rng.choice([0.5, 0.3, 0.7, 0.9, 1.0]))
        ig = int(rng.choice([5, 0, 1, 10, 30])); eg = int(rng.choice([2, 0, 1, 5]))
        extra = ["-coverage", repr(cov), "-identity", repr(idn), "-igap", str(ig), "-egap", str(eg)]
        if ev is not None: extra += ["-evalue", repr(float(ev))]
        for f_ in (ro, oo):
            if os.path.exists(f_): os.remove(f_)
        desc = f"case {seed0}/{case}: nd {nd} nq {nq} len {lo}-{hi} div {div} dirty {dirty} nt {nt} ev {ev} cov {cov} id {idn} ig {ig} eg {eg}"
        db, q = hp.OracleSeqs(dbf, True), hp.OracleSeqs(qf, False)
        best, st = hp.oracle_align(db, q, hp.default_params(n_threads=nt, evalue=None if ev is None else float(ev), coverage=cov,
                                                            identity=idn, igap=ig, egap=eg), out_path=oo)
        if live:
            r = subprocess.run([hp.REF_BIN, "-query", qf, "-db", dbf, "-out", ro, "-n_threads", str(nt)] + extra, capture_output=True, text=True)
            assert r.returncode == 0, (desc, r.stdout[-300:])
            assert hp.parse_align_headers(ro) == hp.parse_align_headers(oo), desc
            if nt == 1:
                assert open(ro, "rb").read() == open(oo, "rb").read(), desc
            summ = [l for l in r.stdout.splitlines() if "from the query were found" in l]
            assert int(summ[0].split()[1]) == st.accepted, desc
        out.append(dict(hp.align_digest(oo, whole=nt == 1), accepted=int(st.accepted), case=desc))
    return out
