"""Threshold sweeps without a GPU: the exported entry point, the host-built per-set and intersection tables, and the
command line's -sweep argument checks, which end the run before any device work."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import helpers as hp

G = os.path.join(hp.ROOT, "tests", "golden")
EXE = os.path.join(hp.ROOT, "bin", "IMSAME")


def test_align_sweep_is_exported(built):
    from imsame_b200 import api
    lib = C.CDLL(api.GPU_SO)
    assert getattr(lib, "imsame_gpu_align_sweep") is not None
    assert "imsame_gpu_align_sweep" in api.SYMBOLS
    hdr = open(os.path.join(hp.ROOT, "include", "imsame_gpu.h")).read()
    assert "#define IMSAME_SWEEP_MAX 16" in hdr and api.SWEEP_MAX == 16


@pytest.mark.parametrize("sets", [
    [(0.5, 0.5)],
    [(0.5, 0.95), (0.5, 0.7), (0.5, 0.85), (0.5, 0.75), (0.5, 0.9), (0.5, 0.8)],
    [(1.0, 0.5), (0.3, 0.5), (0.8, 0.5), (0.5, 0.5), (0.3, 0.5)],
    [(0.5, 0.5), (0.5, 0.5), (0.9, 0.6), (0.2, 1.0), (1.5, 0.33)],
])
def test_sweep_tables_equal_the_single_set_builders(built, sets):
    """per-set tables == imsame_build_lmin / imsame_build_imin of that set; intersection == their elementwise maxima
    (sets in any order, duplicates, the reference's defaults 0.5 / 0.5)"""
    from imsame_b200 import hostlib as H
    cov, idn = [c for c, _ in sets], [i for _, i in sets]
    lmin_sets, imin_sets, lmin_all, imin_all = H.sweep_tables(cov, idn)
    for t, (c, i) in enumerate(sets):
        _, lmin, imin = H.threshold_tables(1e-20, c, i, 1000)
        assert np.array_equal(lmin_sets[t], lmin), t
        assert np.array_equal(imin_sets[t], imin), t
    assert np.array_equal(lmin_all, lmin_sets.max(axis=0))
    assert np.array_equal(imin_all, imin_sets.max(axis=0))


def _run(*extra):
    return subprocess.run([EXE, "-query", os.path.join(G, "dirty.q.fa"), "-db", os.path.join(G, "dirty.db.fa"), *extra],
                          capture_output=True, text=True)


@pytest.mark.parametrize("value,message", [
    ("0.5", "-sweep expects a list of coverage:identity pairs, e.g. -sweep 0.5:0.7,0.5:0.9"),
    ("0.5:0.7,", "-sweep expects a list of coverage:identity pairs, e.g. -sweep 0.5:0.7,0.5:0.9"),
    ("0.5:0.7,0.5:x", "-sweep expects a list of coverage:identity pairs, e.g. -sweep 0.5:0.7,0.5:0.9"),
    (":0.7", "-sweep expects a list of coverage:identity pairs, e.g. -sweep 0.5:0.7,0.5:0.9"),
    ("0.5:0.7:0.9", "-sweep expects a list of coverage:identity pairs, e.g. -sweep 0.5:0.7,0.5:0.9"),
    (",".join(["0.5:0.5"] * 16), "-sweep takes at most 15 coverage:identity pairs"),
    ("0.5:0.7,0:0.5", "Min-coverage must be larger than zero"),
    ("0.5:0.7,-0.1:0.5", "Min-coverage must be larger than zero"),
    ("0.5:0", "Min-identity must be larger than zero"),
    ("0.5:-2", "Min-identity must be larger than zero"),
])
def test_malformed_sweep_list_is_refused_before_any_work(built, value, message):
    """the reference's terror form (message on stdout, exit status 255) and nothing else: no [INFO] line, no GPU"""
    r = _run("-sweep", value)
    assert r.returncode == 255 and r.stdout == f"ERR**** {message} ****\n", r.stdout


@pytest.mark.parametrize("extra,message", [
    (["-gpus", "2"], "-sweep runs on one GPU: it cannot be combined with -gpus above 1"),
    (["-out_rev", "REV"], "-sweep cannot be combined with -out_rev"),
])
def test_sweep_combinations_that_are_refused(built, tmp_path, extra, message):
    extra = [str(tmp_path / "r.align") if e == "REV" else e for e in extra]
    r = _run("-sweep", "0.5:0.7", "-out", str(tmp_path / "f.align"), *extra)
    assert r.returncode == 255 and r.stdout == f"ERR**** {message} ****\n", r.stdout
    assert not os.path.exists(tmp_path / "f.align") and not os.path.exists(tmp_path / "r.align")


def test_sweep_fails_loudly_without_a_gpu(built, tmp_path):
    """no CPU fallback behind -sweep: the reference's error form, exit status 255, every file empty"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    f = tmp_path / "f.align"
    r = _run("-sweep", "0.5:0.7,0.5:0.9", "-out", str(f))
    assert r.returncode == 255 and "ERR**** GPU hot path failed: no usable sm_100 CUDA device" in r.stdout
    assert "from the query were found" not in r.stdout
    assert all(os.path.getsize(p) == 0 for p in (f, f"{f}.1", f"{f}.2"))


def test_sweep_is_not_in_the_reference_help_text(built):
    r = subprocess.run([EXE, "--help"], capture_output=True, text=True)
    assert r.returncode == 1 and "-sweep" not in r.stdout
