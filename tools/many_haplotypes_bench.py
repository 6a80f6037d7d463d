#!/usr/bin/env python3
"""Files -> files on windows with many distinct haplotypes (the block histogram tier), against the oracle.

    python tools/many_haplotypes_bench.py [--transcripts 2000] [--coverage 100] [--dir DIR]

Writes the `manyhap` profile of tests/test_many_haplotypes_emu.py (each somatic variant carried independently by each read,
7 somatic SNVs inside 27 nt of one exon per gene) at the given size into DIR (reused when it is already there), runs
mph_run_somatic and mph_run_normal on it in fresh processes and the oracle on the same files. Prints one JSON line per mode:
wall time, k2_ms / replay_ms / k5_ms from mph_timing, the oracle's wall time, whether the outputs equal the oracle's, the
windows with more than 32 keys in the oracle's window trace (somatic: the windows the block tier takes), the GPU's name and
power limit. The junction merge compares records pairwise inside one warp, so k5_ms grows with the square of the records
of the largest junction."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CHILD = r"""
import json, os, sys, time
sys.path.insert(0, %r)
import microphaser_b200 as m
d, out, mode = sys.argv[1:4]
ctx = m.Context(0)
t0 = time.perf_counter()
args = [os.path.join(d, "reads.bam"), os.path.join(d, "ref.fa"), os.path.join(d, "variants.vcf"), os.path.join(d, "annotation.gtf"),
        os.path.join(out, "out.fa"), os.path.join(out, "out.tsv")]
if mode == "somatic":
    ctx.run_somatic(*args, os.path.join(out, "out.normal.fa"))
else:
    ctx.run_normal(*args)
wall = time.perf_counter() - t0
t = ctx.timing()
ctx.close()
print(json.dumps(dict(wall_s=wall, k2_ms=t["k2_ms"], replay_ms=t["replay_ms"], k5_ms=t["k5_ms"], kernels_ms=t["kernels_ms"])))
""" % ROOT


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--transcripts", type=int, default=2000)
    ap.add_argument("--coverage", type=float, default=100.0)
    ap.add_argument("--dir", default=None, help="where the inputs go (default: a temporary directory); reused if it holds them")
    a = ap.parse_args()
    from microphaser_b200 import build, synth
    from conftest import build_oracle, read_outputs
    from test_many_haplotypes_emu import MANYHAP
    build.build_all()
    oracle = build_oracle()
    d = a.dir or tempfile.mkdtemp(prefix="mph_manyhap_")
    if not os.path.exists(os.path.join(d, "reads.bam")):
        synth.generate(d, synth.Params(seed=2000, **dict(MANYHAP, n_genes=a.transcripts, coverage=a.coverage)))
    work = tempfile.mkdtemp(prefix="mph_manyhap_out_")
    gpu = gpu_info()
    for mode in ("somatic", "normal"):
        o, p = os.path.join(work, mode + "_oracle"), os.path.join(work, mode + "_cuda")
        os.makedirs(o)
        os.makedirs(p)
        env = dict(os.environ)
        trace = os.path.join(work, mode + "_trace.txt")
        if mode == "somatic":
            env["MPH_ORACLE_TRACE"] = trace
        t0 = time.perf_counter()
        cmd = [oracle, mode, os.path.join(d, "reads.bam"), "-r", os.path.join(d, "ref.fa"), "-b", os.path.join(d, "variants.vcf"), "-t", os.path.join(o, "out.tsv")]
        if mode == "somatic":
            cmd += ["-n", os.path.join(o, "out.normal.fa")]
        with open(os.path.join(d, "annotation.gtf")) as gin, open(os.path.join(o, "out.fa"), "wb") as fo:
            ro = subprocess.run(cmd, stdin=gin, stdout=fo, stderr=subprocess.PIPE, env=env)
        oracle_s = time.perf_counter() - t0
        r = subprocess.run([sys.executable, "-c", CHILD, d, p, mode], capture_output=True, text=True)
        line = dict(mode=mode, transcripts=a.transcripts, coverage=a.coverage, gpu=gpu, oracle_s=oracle_s, oracle_rc=ro.returncode)
        if r.returncode != 0:
            line.update(error=r.stderr[-400:])
        else:
            line.update(json.loads(r.stdout.strip().splitlines()[-1]))
            line["equal_to_oracle"] = ro.returncode == 0 and read_outputs(o, mode) == read_outputs(p, mode)
        if mode == "somatic" and os.path.exists(trace):
            keys = [len(t.split("\t")) - 7 for t in open(trace)]
            line.update(trace_windows=len(keys), windows_over_32_keys=sum(k > 32 for k in keys), max_keys=max(keys) if keys else 0)
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
