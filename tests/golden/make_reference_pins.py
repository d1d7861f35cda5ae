#!/usr/bin/env python
"""Writes tests/golden/reference_pins.json: what the unmodified reference tools give on the seeded inputs of the tests
that compare with them (test_oracle_vs_live_reference, test_oracle_fuzz_vs_live_reference,
test_revcomp_fuzz_against_the_reference_tool, test_allvsall_text_filter_samples_reference_workflow_vs_oracle,
test_revcomp_matches_reference_semantics, test_cli_flags_and_errors), as digests of exactly the parts those tests
compare.  The values are taken from the oracle and bin/revComp, which those tests hold equal to the reference; where
oracle/_ref is built the fuzz cases are compared with it on the way.  Run after `make all oracle`."""
import json
import os
import pathlib
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers as hp  # noqa: E402
import synth_cases as sc  # noqa: E402
import test_host_cpu  # noqa: E402
import test_oracle_fuzz  # noqa: E402
import test_oracle_golden  # noqa: E402

ABOUT = ("Digests (sha256) of what the unmodified reference IMSAME, revComp and all_vs_all_metagenomes_IMSAME.sh give on "
         "the seeded inputs of the tests that compare with them; those tests compare with these values where the "
         "reference is not built.  Recorded by make_reference_pins.py from the oracle (oracle/imsame_oracle.c) and "
         "bin/revComp (imsame_b200/host/fasta.c), whose sources are unchanged since the same tests last found them equal "
         "to the reference binaries on these inputs.  revcomp_fuzz: the few cases on which the reference revComp died on "
         "a signal were never compared with it; they hold bin/revComp's result.")


def main():
    live = hp.have_reference()
    pins = {"about": ABOUT}
    with tempfile.TemporaryDirectory() as d:
        pins["oracle_vs_live_reference"] = {}
        for seed, div, nt in test_oracle_golden.LIVE_CASES:
            _, _, orc_out = test_oracle_golden.live_case(seed, div, nt, d)
            pins["oracle_vs_live_reference"][f"{seed}/{div}/{nt}"] = hp.align_digest(orc_out, whole=nt == 1)
        pins["oracle_fuzz"] = {str(s): test_oracle_fuzz.fuzz_cases(s, d, live) for s in (11, 12)}
        pins["revcomp_fuzz"] = test_host_cpu.revcomp_fuzz(d, os.path.exists(hp.REF_REVCOMP))
        samples = os.path.join(d, "samples")
        os.makedirs(samples)
        sc.write_allvsall_filter_samples(pathlib.Path(samples))
        p = hp.default_params(n_threads=2, coverage=0.5, identity=0.5)
        q = hp.OracleSeqs(os.path.join(samples, "s0.fasta"), False)
        pins["allvsall_text_filter_samples"] = {}
        for y in ("s1", "s2", "s3"):
            for rev in (0, 1):
                dbf = os.path.join(samples, f"{y}.fasta")
                if rev:
                    subprocess.check_call([os.path.join(ROOT, "bin", "revComp"), dbf, os.path.join(d, "r.fasta")],
                                          stdout=subprocess.DEVNULL)
                    dbf = os.path.join(d, "r.fasta")
                oo = os.path.join(d, "orc.align")
                hp.oracle_align(hp.OracleSeqs(dbf, True), q, p, out_path=oo)
                pins["allvsall_text_filter_samples"][f"s0-{y}{'.r' if rev else ''}.align"] = hp.align_digest(oo, lines=True)
        o = os.path.join(d, "dirty.r.fa")
        subprocess.check_call([os.path.join(ROOT, "bin", "revComp"), os.path.join(HERE, "dirty.db.fa"), o])
        pins["revcomp_dirty_db"] = hp.sha(open(o, "rb").read())
    qf = os.path.join(HERE, "dirty.q.fa")
    pins["cli_error_forms"] = []
    for args in (["--help"], ["-query", "nope"], ["-query", qf, "-db", qf, "-identity", "-1"]):
        a = subprocess.run([os.path.join(ROOT, "bin", "IMSAME")] + args, capture_output=True, text=True)
        pins["cli_error_forms"].append([a.returncode, hp.sha(a.stdout.encode())])
    with open(os.path.join(HERE, "reference_pins.json"), "w") as f:
        json.dump(pins, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
