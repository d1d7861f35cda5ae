#!/usr/bin/env python
"""cfg4 (BASELINE.json configs[3]: 8 synthetic metagenome samples of 100 k reads x 150 bp, the seeded pool of
tools/allvsall_bench.py) at the six identity thresholds of cfg5 (configs[4]: coverage 0.5, identity 0.70 .. 0.95):
one bin/IMSAME_allvsall -sweep run against six separate IMSAME_allvsall runs, in the same call.  Every file of the sweep
run is compared byte for byte with the separate runs' (entry i's X-Y[.r].align.i with the X-Y[.r].align of the run at
that threshold); prints the wall times, the card and its power limit.
usage: python tools/allvsall_sweep_bench.py [--samples 8] [--reads 100000] [--repeats 1]"""
import argparse, filecmp, os, shutil, subprocess, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from imsame_b200 import hostlib as H  # noqa: E402
ap = argparse.ArgumentParser()
ap.add_argument("--samples", type=int, default=8)
ap.add_argument("--reads", type=int, default=100000)
ap.add_argument("--threads", type=int, default=os.cpu_count() or 8)
ap.add_argument("--repeats", type=int, default=1)
a = ap.parse_args()
SETS = [("0.5", i) for i in ("0.70", "0.75", "0.80", "0.85", "0.90", "0.95")]
EXE = os.path.join(ROOT, "bin", "IMSAME_allvsall")
d = tempfile.mkdtemp(prefix="imsame_avall_sweep_")
sd = os.path.join(d, "samples")
os.makedirs(sd)
pool = H.SynthPool(4001, 40, 500_000)
for s in range(a.samples):
    H.write_fasta(os.path.join(sd, f"m{s}.fasta"), pool.db_reads(s * a.reads, a.reads, 150), a.reads, 150, "r")
pool.close()
smi = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
print("cards (index, name, power limit):")
print(smi.stdout.strip() or smi.stderr.strip())
print(f"{a.samples} samples x {a.reads} reads x 150 bp, {a.samples * (a.samples - 1)} units, -n_threads {a.threads}, "
      f"sets {' '.join(c + ':' + i for c, i in SETS)}")


def run(out, cov, idn, extra=()):
    os.makedirs(out)
    t = time.time()
    r = subprocess.run([EXE, sd, cov, idn, str(a.threads), "fasta", out] + list(extra), capture_output=True, text=True)
    dt = time.time() - t
    if r.returncode:
        sys.exit(f"{out}: rc {r.returncode}: {r.stdout[-500:]}{r.stderr[-500:]}")
    return dt


t_sweep, t_sep, ok = [], [], True
for rep in range(a.repeats):
    # the sweep's main thresholds are the first set; entries 1..5 the others
    so = os.path.join(d, f"sweep{rep}")
    t_sweep.append(run(so, *SETS[0], ["-sweep", ",".join(f"{c}:{i}" for c, i in SETS[1:])]))
    seps, t = [], 0.0
    for k, (c, i) in enumerate(SETS):
        seps.append(os.path.join(d, f"sep{rep}_{k}"))
        t += run(seps[-1], c, i)
    t_sep.append(t)
    names = sorted(os.listdir(seps[0]))
    same = sorted(os.listdir(so)) == sorted(names + [f"{n}.{k}" for n in names for k in range(1, len(SETS))])
    for n in names:
        for k, sep in enumerate(seps):
            same &= filecmp.cmp(os.path.join(so, n + (f".{k}" if k else "")), os.path.join(sep, n), shallow=False)
    ok &= same
    size = sum(os.path.getsize(os.path.join(so, n)) for n in os.listdir(so))
    print(f"run {rep}: one -sweep run {t_sweep[-1]:.2f} s wall, six separate runs {t:.2f} s wall; "
          f"{len(os.listdir(so))} files, {size / 1e6:.0f} MB; all files byte-identical: {same}")
    sys.stdout.flush()
    for p in [so] + seps:
        shutil.rmtree(p)
ms, mp = sorted(t_sweep)[len(t_sweep) // 2], sorted(t_sep)[len(t_sep) // 2]
print(f"medians over {a.repeats} run(s): -sweep {ms:.2f} s, separate {mp:.2f} s, speed-up {mp / ms:.2f}x; "
      f"all files identical: {ok}")
shutil.rmtree(d, ignore_errors=True)
sys.exit(0 if ok else 1)
