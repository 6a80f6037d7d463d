"""Windows with more distinct haplotype keys than a warp table (32) holds, through the CPU emulator: the serial replay's
fold of such windows in the key arena, the host residue's key buffers and junctions with more than 255 merged records,
against the oracle. The CUDA path runs the same inputs in tests/test_gpu_many_haplotypes.py (-m gpu)."""
import collections
import hashlib
import os
import subprocess
import sys

import pytest

from conftest import ROOT, read_outputs, run_cli

sys.path.insert(0, ROOT)
from microphaser_b200 import synth  # noqa: E402

# every somatic variant carried independently by each read, plus 7 somatic SNVs inside 27 nt of one exon per gene
MANYHAP = dict(independent_somatic=True, hotspot_per_gene=7, somatic_per_kb=40.0, germline_per_kb=8.0, coverage=100.0, n_genes=3)
MANYHAP_PROFILES = {
    "manyhap": dict(MANYHAP),
    "manyhap_carry": dict(MANYHAP, intron_len=(15, 80), indel_frac=0.1),  # observations survive into the next exon: serial replay
    "manyhap_fs": dict(MANYHAP, indel_frac=0.3, frameshift_ok=True),    # frameshifting indels: host-class transcripts
    # short exons, a denser hotspot: both windows of a splice junction carry dozens of keys
    "manyhap_junction": dict(MANYHAP, hotspot_per_gene=9, somatic_per_kb=60.0, germline_per_kb=10.0, coverage=150.0, n_genes=4, exon_len=(28, 40)),
}
SEEDS = (6, 11)
# 20 somatic SNVs inside one window, each read carrying each of them independently, at a depth that gives more than
# MPH_BLOCK_KEYS (4096) distinct allele patterns in that window
LIMIT = dict(independent_somatic=True, hotspot_per_gene=20, somatic_per_kb=0.0, germline_per_kb=0.0, coverage=12000.0, n_genes=1, exons=(2, 2),
             exon_len=(60, 80), variants_in_introns=False)
LIMIT_REPLAY = dict(LIMIT, intron_len=(15, 80))  # the same through the serial replay (an intron shorter than a read)
LIMIT_MSG = b"more than 4096 distinct haplotypes in one window"


def make_input(tmp_path, profile, seed):
    d = str(tmp_path / ("in_%s_%d" % (profile, seed)))
    if not os.path.exists(d):
        synth.generate(d, synth.Params(seed=seed, **MANYHAP_PROFILES[profile]))
    return d


def oracle_trace(oracle_bin, d, tmp_path):
    """The oracle's MPH_ORACLE_TRACE window lines: (transcript, frame, keys)."""
    o = tmp_path / "trace_out"
    o.mkdir(exist_ok=True)
    tr = str(tmp_path / "trace.txt")
    env = dict(os.environ, MPH_ORACLE_TRACE=tr)
    with open(os.path.join(d, "annotation.gtf")) as gin, open(o / "out.fa", "wb") as fo:
        r = subprocess.run([oracle_bin, "somatic", os.path.join(d, "reads.bam"), "-r", os.path.join(d, "ref.fa"), "-b", os.path.join(d, "variants.vcf"),
                            "-t", str(o / "out.tsv"), "-n", str(o / "out.normal.fa")], stdin=gin, stdout=fo, stderr=subprocess.PIPE, env=env)
    assert r.returncode == 0, r.stderr.decode()[-300:]
    out = []
    for line in open(tr):
        f = line.rstrip("\n").split("\t")
        out.append((f[1], int(f[4]), len(f) - 7))
    return out


def short_intron_transcripts(d, read_len=100):
    """Transcripts with an intron shorter than a read: reads span it, so the transcript goes through the serial replay."""
    exons = {}
    for line in open(os.path.join(d, "annotation.gtf")):
        t = line.split("\t")
        if len(t) > 8 and t[2] == "exon":
            tid = t[8].split('transcript_id "')[1].split('"')[0]
            exons.setdefault(tid, []).append((int(t[3]), int(t[4])))
    out = set()
    for tid, ex in exons.items():
        ex.sort()
        if any(b[0] - a[1] - 1 < read_len for a, b in zip(ex, ex[1:])):
            out.add(tid)
    return out


def junction_records(d, tsv, window_len=27):
    """Records of the oracle's TSV per (transcript, exon end) whose window straddles that end: the records of a splice
    junction's merge (a window's own records lie inside one exon)."""
    exons = collections.defaultdict(list)
    for line in open(os.path.join(d, "annotation.gtf")):
        t = line.split("\t")
        if len(t) > 8 and t[2] == "exon":
            exons[t[8].split('transcript_id "')[1].split('"')[0]].append((int(t[3]) - 1, int(t[4])))
    out = collections.Counter()
    for line in list(open(tsv))[1:]:
        f = line.split("\t")
        tx, off = f[1], int(f[5])
        if any(s - 1 <= off and off + window_len <= e + 1 for s, e in exons[tx]):
            continue
        out[(tx, min((e for s, e in exons[tx] if s - 1 <= off < e + 1), default=None))] += 1
    return out


@pytest.mark.parametrize("seed", SEEDS)
def test_inputs_reach_more_than_32_keys(oracle_bin, seed, tmp_path):
    """Each profile does what it is for, as the oracle's window trace and output show."""
    for profile in MANYHAP_PROFILES:
        d = make_input(tmp_path, profile, seed)
        wins = oracle_trace(oracle_bin, d, tmp_path)
        assert max(k for _, _, k in wins) > 32, profile
        if profile == "manyhap_carry":
            replayed = short_intron_transcripts(d)
            assert any(t in replayed and k > 32 for t, _, k in wins), "no replayed window with more than 32 keys"
        if profile == "manyhap_fs":
            assert any(f > 0 and k > 32 for _, f, k in wins), "no frameshift window with more than 32 keys"
        if profile == "manyhap_junction":
            o = tmp_path / ("junction_%d" % seed)
            o.mkdir()
            assert run_cli(oracle_bin, d, str(o)).returncode == 0
            assert max(junction_records(d, str(o / "out.tsv")).values()) > 255


@pytest.mark.parametrize("mode", ["somatic", "normal"])
@pytest.mark.parametrize("profile", list(MANYHAP_PROFILES))
@pytest.mark.parametrize("seed", SEEDS)
def test_emulated_path_matches_oracle_with_many_keys(emu_bin, oracle_bin, profile, seed, mode, tmp_path):
    d = make_input(tmp_path, profile, seed)
    o, p = tmp_path / "o", tmp_path / "p"
    o.mkdir()
    p.mkdir()
    ro = run_cli(oracle_bin, d, str(o), subcommand=mode)
    rp = run_cli(emu_bin, d, str(p), subcommand=mode)
    assert ro.returncode == 0, ro.stderr.decode()[-300:]
    assert rp.returncode == 0, rp.stderr.decode()[-300:]
    assert read_outputs(str(o), mode) == read_outputs(str(p), mode)


@pytest.mark.parametrize("mode", ["somatic", "normal"])
def test_more_than_4096_keys_is_unsupported(emu_bin, mode, tmp_path):
    """The serial replay's fold keeps the block tier's bound (the emulator's closed form has no key table to bound)."""
    d = str(tmp_path / "in")
    synth.generate(d, synth.Params(seed=21, **LIMIT_REPLAY))
    p = tmp_path / "p"
    p.mkdir()
    r = run_cli(emu_bin, d, str(p), subcommand=mode)
    assert r.returncode == 3, r.stderr.decode()[-300:]
    assert LIMIT_MSG in r.stderr


# sha256 over (file name, bytes) of everything synth.generate writes, per tests/test_emu_parity.py PROFILES entry at seed
# 11 * 7919 + len(name), 3 genes, 25x: the new generator parameters at their defaults draw the same random numbers as before
GENERATOR_HASHES = {
    "snv": "5ad317e940a35c46",
    "indel": "98234881194d8212",
    "geom": "d0b3e729977d0ec9",
    "dense": "dc1e4b71f491f57f",
    "fs": "d0cae48f489f907c",
    "multi": "a157c240ef1dc756",
    "carry": "3fc67f21b8e352ef",
    "anti": "b356dcf0849755a7",
    "dups": "39606365652380e0",
}


def test_generator_unchanged_at_defaults(tmp_path):
    from test_emu_parity import PROFILES
    assert set(PROFILES) == set(GENERATOR_HASHES)
    for name, kw in PROFILES.items():
        kw = dict(kw, seed=11 * 7919 + len(name), n_genes=3, coverage=25.0)
        d = str(tmp_path / name)
        synth.generate(d, synth.Params(**kw))
        h = hashlib.sha256()
        for f in sorted(os.listdir(d)):
            h.update(f.encode())
            h.update(open(os.path.join(d, f), "rb").read())
        assert h.hexdigest()[:16] == GENERATOR_HASHES[name], name
