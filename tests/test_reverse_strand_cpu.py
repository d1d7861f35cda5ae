"""The reverse strand of the resident database without a GPU: the device functions of imsame_gpu_db_revcomp
(csrc/revcomp.cuh) emulated on random multi-segment layouts, and the command line's -out_rev on a machine without
an sm_100 device."""
import os
import subprocess

import pytest

import helpers as hp

G = os.path.join(hp.ROOT, "tests", "golden")
EXE = os.path.join(hp.ROOT, "bin", "IMSAME")


@pytest.mark.parametrize("seed", [1, 2])
def test_segment_mirror_on_cpu(built, seed, tmp_path):
    """revcomp_word + the segment mirror arithmetic against a plain reverse complement of the concatenated reads, laid
    out into segments as the loader would: fixed and ragged reads, totals that are no multiple of 16, one-read
    segments, word breaks at read and segment starts, and the mirror applied twice against the forward layout"""
    exe = str(tmp_path / "revcomp_emul")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(hp.ROOT, "tests", "emul", "revcomp_emul.cpp")])
    r = subprocess.run([exe, "3000", str(seed)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:]
    assert "0 mismatches" in r.stdout


def test_out_rev_fails_loudly_without_a_gpu(built, tmp_path):
    """no CPU fallback behind -out_rev: the reference's error form, exit status 255, no record in either file"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    out, rev = tmp_path / "f.align", tmp_path / "r.align"
    r = subprocess.run([EXE, "-query", os.path.join(G, "dirty.q.fa"), "-db", os.path.join(G, "dirty.db.fa"), "-out", str(out),
                        "-out_rev", str(rev)], capture_output=True, text=True)
    assert r.returncode == 255 and "ERR**** GPU hot path failed: no usable sm_100 CUDA device" in r.stdout
    assert "from the query were found" not in r.stdout
    assert os.path.getsize(out) == 0 and os.path.getsize(rev) == 0


def test_out_rev_unopenable_path(built, tmp_path):
    """the reverse-strand file is opened before any work; a path that cannot be opened ends the run right there"""
    r = subprocess.run([EXE, "-query", os.path.join(G, "dirty.q.fa"), "-db", os.path.join(G, "dirty.db.fa"),
                        "-out_rev", str(tmp_path / "no" / "such" / "dir" / "r.align")], capture_output=True, text=True)
    assert r.returncode == 255
    assert r.stdout == "ERR**** Could not open the reverse-strand output file ****\n"


def test_out_rev_is_not_in_the_reference_help_text(built):
    r = subprocess.run([EXE, "--help"], capture_output=True, text=True)
    assert r.returncode == 1 and "-out_rev" not in r.stdout
