#!/usr/bin/env python3
"""bench.py — phased windows/s of the per-window phasing hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload exome|chr22|hypermutated|normal|filter] [--dump-outputs DIR]

Default workload (config.workload): one whole-exome-shaped shard per GPU — BASELINE.json configs[2]
("synthetic whole exome (~20k transcripts), 100x tumor BAM, somatic mode"): 20 000 single-transcript
genes x 8 CDS exons, 150 bp reads at 100x, 1 germline + 1 somatic SNV per kb. It fits one GPU; its device arrays
(~0.6 GB) are far larger than the 126 MB L2 and a 256 MB buffer is rewritten between steps all the same. Weak scaling: every rank phases its own
shard (different seed), there is no collective on the data path; ranks only meet at the timing barrier.
The other workloads are the remaining synthetic configs of BASELINE.json (chr22 exome, hypermutated tumour,
`normal` healthy peptidome, `filter` set probe).

A step = one pass of the hot path over the shard.
  value : windows/s with the packed shard resident in HBM (all kernels of the path, CUDA events on the
          library's stream, max over ranks).
  e2e   : windows/s through the C ABI call mph_phase_batch with pinned HOST buffers: H2D copy, kernels,
          D2H copy of the ordered records (plus the host residue of the irregular transcripts).
  e2e_files : files -> files on a bounded slice of the workload: BAM / VCF / GTF / FASTA in, FASTA / TSV out
          through mph_run_somatic (ingest, packing, phasing, text rendering and writing all on the clock),
          next to the CPU oracle on the same files.
  parity_checked : records of the benched batch that were compared byte for byte with the oracle's output.
  roofline     : dominant kernel vs the measured HBM copy bandwidth (MEASURED_PEAKS.json); its kernel times come from a
          second pass of the same steps with every kernel alone on one stream (in the timed loop the serial replay of
          the irregular transcripts runs beside K2 / K3 / K5 on a second stream).
  cpu_baseline : the CPU oracle (a restatement of the reference's Rust code, which cannot be built
          here — no cargo/rustc) on one core over a bounded sample of the same workload.
`--impl reference` times that oracle on all host cores instead.

`--dump-outputs DIR` writes what the last timed step computed (rank 0) as DIR/<name>.npy: the records of
mph_phase_resident (a fixed, seeded sample when there are more than DUMP_RECORDS; every field, strings as byte
values with a length per record) or the hit flags of the filter probe. The inputs are seeded, so two builds
can be compared array for array.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "exome": dict(n_transcripts=20000, coverage=100.0, germline_per_kb=1.0, somatic_per_kb=1.0, ins_var_frac=0.0, del_var_frac=0.0, mode="somatic",
                  desc="synthetic whole exome shard per GPU (BASELINE.json configs[2]): 20000 transcripts x 8 exons, 100x, 150 bp, 1+1 SNV/kb"),
    "chr22": dict(n_transcripts=450, coverage=30.0, germline_per_kb=1.0, somatic_per_kb=1.0, ins_var_frac=0.0, del_var_frac=0.0, mode="somatic",
                  desc="synthetic chr22 exome (BASELINE.json configs[1]): 450 transcripts x 8 exons, 30x, 150 bp, 1+1 SNV/kb"),
    "hypermutated": dict(n_transcripts=4000, coverage=100.0, germline_per_kb=1.0, somatic_per_kb=10.0, ins_var_frac=0.1, del_var_frac=0.1, mode="somatic",
                         desc="synthetic hypermutated tumour (BASELINE.json configs[3]): 4000 transcripts x 8 exons, 100x, 150 bp, 1 germline + 10 somatic variants/kb, 10 % insertions + 10 % deletions"),
    "normal": dict(n_transcripts=5000, coverage=30.0, germline_per_kb=1.0, somatic_per_kb=1.0, ins_var_frac=0.0, del_var_frac=0.0, mode="normal",
                   desc="synthetic healthy peptidome, `normal` mode (BASELINE.json configs[4]a): 5000 transcripts x 8 exons, 30x, 150 bp, every window is a record"),
    "filter": dict(desc="`filter` set probe (BASELINE.json configs[4]b): 1 M neopeptides (9-mers) against a normal peptidome of 8 M distinct 9-mers", mode="filter"),
}
SEED = 0x4D500003
METRIC = "phased peptide windows/sec"
UNIT = "windows/s"


def config_of(name):
    """The `config` dict of both arms (identical by construction)."""
    w = WORKLOADS[name]
    big = name in ("exome", "hypermutated", "normal", "filter")
    return {"workload": w["desc"],
            "l2": ("a 256 MB buffer is rewritten between steps (L2 flush); the shard's device arrays exceed the 126 MB L2 anyway" if big
                   else "inputs fit in L2: a 256 MB buffer is rewritten between steps (L2 flush)"),
            "sharding": "one shard per GPU by gene range, no collective"}


def synth_kw(name):
    return {k: v for k, v in WORKLOADS[name].items() if k != "desc"}


def clocks_sampler(device, stop, out):
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    try:
        p = subprocess.Popen(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100", "-i", str(device)],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return
    def reader():
        for line in p.stdout:
            out.append(line.strip())
    t = threading.Thread(target=reader, daemon=True)
    t.start()
    stop.wait()
    p.terminate()
    t.join(timeout=2)


def summarize_clocks(lines):
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for l in lines:
        f = [x.strip() for x in l.split(",")]
        if len(f) < 6:
            continue
        try:
            sm.append(float(f[0]))
            mx.append(float(f[1]))
        except ValueError:
            continue
        for n, v in zip(names, f[2:6]):
            if v.lower().startswith("active"):
                reasons.add(n)
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
    return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons)}


def ensure_oracle():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True)


def write_sample_files(name, n_transcripts, seed, d):
    """The first `n_transcripts` transcripts of the workload as files, written by oracle/_build/mph_synth_files: a stand-alone
    tool built from the generator's host-only header, so the reference arm never loads the CUDA library."""
    kw = synth_kw(name)
    os.makedirs(d, exist_ok=True)
    t = time.time()
    subprocess.run([os.path.join(ROOT, "oracle", "_build", "mph_synth_files"), d, str(seed), str(n_transcripts), str(kw["coverage"]),
                    str(kw["germline_per_kb"]), str(kw["somatic_per_kb"]), str(kw["ins_var_frac"]), str(kw["del_var_frac"])],
                   check=True, stdout=subprocess.DEVNULL)
    return time.time() - t


def run_oracle(d, tag, mode="somatic"):
    stats = os.path.join(d, "stats_%s.json" % tag)
    env = dict(os.environ, MPH_ORACLE_STATS=stats)
    oracle = os.path.join(ROOT, "oracle", "_build", "mph_oracle")
    cmd = [oracle, mode, os.path.join(d, "reads.bam"), "-r", os.path.join(d, "ref.fa"), "-b", os.path.join(d, "variants.vcf"), "-t",
           os.path.join(d, "o_%s.tsv" % tag)]
    if mode == "somatic":
        cmd += ["-n", os.path.join(d, "o_%s.n.fa" % tag)]
    with open(os.path.join(d, "annotation.gtf")) as gin, open(os.path.join(d, "o_%s.fa" % tag), "wb") as fo:
        p = subprocess.Popen(cmd, stdin=gin, stdout=fo, stderr=subprocess.DEVNULL, env=env)
    return p, stats


def reference_arm(args, rank, world):
    """The reference's CPU implementation of the path (oracle port) on all host cores."""
    if rank != 0:
        return
    ensure_oracle()
    name = args.workload
    if name == "filter":
        print(json.dumps({"impl": "reference", "unavailable": "the filter probe workload has no file-level oracle arm; see tests/test_gpu_peptides.py"}))
        return
    w = WORKLOADS[name]
    cores = os.cpu_count() or 1
    sample_tx = min(w["n_transcripts"], 200)
    with tempfile.TemporaryDirectory() as tmp:
        d = os.path.join(tmp, "sample")
        write_sample_files(name, sample_tx, SEED, d)
        per_step = []
        windows = 0
        for step in range(args.warmup + args.steps):
            t0 = time.time()
            procs = [run_oracle(d, "p%d" % i, w["mode"]) for i in range(cores)]
            for p, _ in procs:
                p.wait()
            dt = time.time() - t0
            windows = sum(json.load(open(s))["windows"] for _, s in procs)
            if step >= args.warmup:
                per_step.append(dt)
        ms = 1000.0 * sum(per_step) / len(per_step)
        value = windows / (ms / 1000.0)
    sample = "first %d of %d transcripts of the workload (%d main-ORF windows), one oracle process per core on the same sample, files -> files" % (
        sample_tx, w["n_transcripts"], windows // cores)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": config_of(name),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def shard_seed(rank):
    """Weak scaling: every rank phases its own whole-exome-shaped shard (a different gene range of a larger cohort)."""
    return SEED + rank


def aggregate_over_ranks(dist, device, dev_ms, e2e_ms, windows, read_windows):
    """Time = max over ranks, work = sum over ranks (no other communication happens on this path)."""
    import torch
    vals = torch.tensor([dev_ms, e2e_ms, float(windows), float(read_windows)], dtype=torch.float64, device=device)
    if dist is None:
        return dev_ms, e2e_ms, float(windows), float(read_windows)
    mx = vals.clone()
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    sm = vals.clone()
    dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    return mx[0].item(), mx[1].item(), sm[2].item(), sm[3].item()


KERNEL_KEYS = ("k1_ms", "replay_ms", "k2_ms", "k3_ms", "k4_ms", "k5_ms")

DUMP_RECORDS = 16384  # records sampled for --dump-outputs; keeps the dump of every workload well under DUMP_LIMIT
DUMP_LIMIT = 64 << 20


def write_dump(out_dir, arrays):
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d byte limit" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def dump_records(res, out_dir):
    """Every field of the records a caller of the path receives (mph_record): numbers as float64, each string field as
    its bytes (float32, concatenated) plus <field>_len (float64, -1 for NULL). More than DUMP_RECORDS records are sampled
    with a fixed seed; record_index holds the sampled positions and n_records the full count."""
    import ctypes
    import numpy as np
    import microphaser_b200 as m
    n = len(res)
    idx = np.arange(n) if n <= DUMP_RECORDS else np.sort(np.random.default_rng(SEED).choice(n, DUMP_RECORDS, replace=False))
    recs = [res.record(int(i)) for i in idx]
    arrays = {"n_records": np.array([n], dtype=np.float64), "record_index": idx.astype(np.float64)}
    for f, typ in m.Record._fields_:
        vals = [r[f] for r in recs]
        if typ is ctypes.c_char_p:
            raw = [None if v is None else v.encode() for v in vals]
            arrays[f + "_len"] = np.array([-1 if b is None else len(b) for b in raw], dtype=np.float64)
            arrays[f] = np.frombuffer(b"".join(b or b"" for b in raw), dtype=np.uint8).astype(np.float32)
        else:
            arrays[f] = np.array(vals, dtype=np.float64)
    write_dump(out_dir, arrays)


def filter_workload(args, rank, local_rank, world, dist, barrier):
    """BASELINE.json configs[4]b: ref_set.contains(peptide) for 1 M neopeptides (reference src/peptides.rs:502,684)."""
    import numpy as np
    import torch
    import microphaser_b200 as m
    ctx = m.Context(local_rank)
    rng = np.random.default_rng(SEED + rank)
    aa = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWY", dtype=np.uint8)
    n_ref, n_q, k = 8_000_000, 1_000_000, 9
    ref = aa[rng.integers(0, 20, size=(n_ref, k))]
    queries = aa[rng.integers(0, 20, size=(n_q, k))]
    queries[: n_q // 4] = ref[rng.integers(0, n_ref, size=n_q // 4)]  # a quarter of the queries are members
    ctx.set_load(ref, k)
    ms, kern = [], []
    hits = None
    for i in range(args.warmup + args.steps):
        barrier()
        t0 = time.perf_counter()
        hits = ctx.set_probe(queries, k)
        dt = (time.perf_counter() - t0) * 1000.0
        if i >= args.warmup:
            ms.append(dt)
            kern.append(ctx.timing()["k1_ms"])
    if args.dump_outputs and rank == 0:
        write_dump(args.dump_outputs, {"hits": hits.astype(np.float32)})
    ref_set = set(map(bytes, ref[:200000]))
    sample = queries[:5000]
    for q, h in zip(sample, hits[:5000]):
        if bytes(q) in ref_set:
            assert h == 1, "a member of the reference set was not found"
    assert int(hits[: n_q // 4].sum()) == n_q // 4
    step_ms, k_ms = sum(ms) / len(ms), sum(kern) / len(kern)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = json.load(open(peaks_path))["hbm_gbs"] if os.path.exists(peaks_path) else 6650.0
    alg = n_q * (k + 1) + n_q * 32  # query bytes in, hit byte out, one 32 B sector of the table per probe
    achieved = alg / (k_ms / 1000.0) / 1e9 if k_ms > 0 else 0.0
    if rank == 0:
        print(json.dumps({
            "metric": "filter peptides/sec", "value": n_q * world / (k_ms / 1000.0) if k_ms > 0 else None, "unit": "peptides/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": k_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic", "config": config_of("filter"),
            "e2e": {"value": n_q * world / (step_ms / 1000.0), "unit": "peptides/s", "h2d_bytes_per_step": n_q * k, "d2h_bytes_per_step": n_q, "ms_per_step": step_ms},
            "gpu_launches": args.steps,
            "roofline": {"bound": "hbm", "kernel": "k_set_probe", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "note": "random 32 B sector reads of a 256 MB open-addressing table: sector-bound, not streaming"},
            "cpu_baseline": None}))
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="exome", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-sample-transcripts", type=int, default=1000)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle run (and with it the parity check and e2e_files)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="end-to-end calls to time (default: --steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path; the reference arm writes files only")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import microphaser_b200 as m
    from microphaser_b200 import build as mb
    mb.build_all()
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    if args.workload == "filter":
        filter_workload(args, rank, local_rank, world, dist, barrier)
        if dist is not None:
            dist.destroy_process_group()
        return

    name = args.workload
    w = WORKLOADS[name]
    kw = synth_kw(name)
    mode = kw["mode"]
    # the few host threads the call still uses (host-class transcripts, record copies): every rank gets its share of the cores
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    if local_world > 1:
        os.environ.setdefault("MPH_HOST_THREADS", str(max(1, (os.cpu_count() or 1) // local_world)))
    ctx = m.Context(local_rank)
    t0 = time.time()
    batch = m.Batch.synthetic(seed=shard_seed(rank), pin=True, **kw)
    gen_s = time.time() - t0
    view = batch.view()

    # ---- resident: kernels only, CUDA events on the library's stream
    ctx.upload(batch)
    # one complete pass first: mph_phase_collect re-runs the kernels with larger arenas when the first attempt ran out of
    # record / key space (a fresh context starts small), and mph_phase_resident alone never looks at the overflow flag - a
    # timed loop on undersized arenas would skip part of the junction merges
    ctx.phase_resident()
    ctx.collect().close()
    # L2 flush between steps (a buffer twice the 126 MB L2 is rewritten): what crosses the bus is a fraction of what the
    # kernels read (the exome shard's decoded arrays are ~0.6 GB), but every workload is timed the same, cold-L2 way
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:%d" % local_rank)

    def l2_flush():
        if flush is not None:
            flush.add_(1)
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        l2_flush()
        ctx.phase_resident()
    clk_lines, stop = [], threading.Event()
    sampler = threading.Thread(target=clocks_sampler, args=(local_rank, stop, clk_lines), daemon=True)
    sampler.start()
    barrier()
    per_kernel = {k: 0.0 for k in KERNEL_KEYS}
    chain_ms = 0.0
    launches_timed = 0
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        l2_flush()
        ctx.phase_resident()
        t = ctx.timing()
        chain_ms += t["kernels_ms"]  # CUDA events around the whole kernel chain (k_replay overlaps K2 on a second stream)
        launches_timed += int(t["kernel_launches"])  # counted at the launch sites of the library
        for k in per_kernel:
            per_kernel[k] += t[k]
    barrier()
    wall_res = time.perf_counter() - wall0
    res = ctx.collect()
    t_res = ctx.timing()
    n_records = len(res)
    if args.dump_outputs and rank == 0:
        dump_records(res, args.dump_outputs)
    res.close()
    windows, read_windows = t_res["windows"], t_res["read_windows"]
    dev_ms = chain_ms / args.steps
    # ---- the same steps once more with every kernel on one stream (MPH_SIDE_REPLAY=0): in the timed loop above the serial
    # replay of the irregular transcripts runs beside K2 / K3 / K5 on a second stream, which shortens the step but stretches
    # the kernels it overlaps; the roofline line wants the dominant kernel timed alone (burst peak), so it is taken here
    per_kernel_overlapped = dict(per_kernel)
    side_prev = os.environ.get("MPH_SIDE_REPLAY")
    os.environ["MPH_SIDE_REPLAY"] = "0"
    per_kernel = {k: 0.0 for k in KERNEL_KEYS}
    serial_chain_ms = 0.0
    l2_flush()
    ctx.phase_resident()
    for _ in range(args.steps):
        l2_flush()
        ctx.phase_resident()
        t = ctx.timing()
        serial_chain_ms += t["kernels_ms"]
        for k in per_kernel:
            per_kernel[k] += t[k]
    if side_prev is None:
        del os.environ["MPH_SIDE_REPLAY"]
    else:
        os.environ["MPH_SIDE_REPLAY"] = side_prev

    # ---- end to end through the C ABI: pinned host buffers -> ordered records
    n_e2e = args.e2e_steps or args.steps
    e2e_ms, h2d_b, d2h_b = [], 0, 0
    stage = {k: 0.0 for k in ("h2d_ms", "d2h_ms", "residue_ms")}
    last = None
    for i in range(1 + n_e2e):
        barrier()
        w0 = time.perf_counter()
        r = ctx.phase_batch(batch)
        dt = (time.perf_counter() - w0) * 1000.0
        t = ctx.timing()
        if last is not None:
            last.close()
        last = r
        if i > 0:
            e2e_ms.append(dt)
            h2d_b, d2h_b = t["h2d_bytes"], t["d2h_bytes"]
            for k in stage:
                stage[k] += t[k] / n_e2e
    stop.set()
    sampler.join(timeout=3)
    e2e_step_ms = sum(e2e_ms) / len(e2e_ms)

    # ---- max over ranks
    dev_ms_max, e2e_ms_max, windows_all, rw_all = aggregate_over_ranks(dist, "cuda:%d" % local_rank, dev_ms, e2e_step_ms, windows, read_windows)
    if rank != 0:
        last.close()
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (algorithmic = compulsory bytes of this design, DESIGN.md §5)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    n_reads, n_win, n_seg, n_chunk = view.n_reads, view.n_windows, view.n_segments, view.n_chunks
    n_special = float(view.n_variant_reads)  # side-table entries: reads that overlap a variant
    alg = {
        # zero-fill of flag / nv for every read (2 B), then per side-table entry: entry in (21 B), start / end (8 B), one base
        # sector + one quality sector (64 B), S / B / flag / vlo / nv / index out (26 B)
        "k1_ms": n_reads * 2 + n_special * (21 + 8 + 64 + 26) + view.n_vars * 16,
        # K2a: start, end, call flag, host flag per (segment, read) pair (10 B) + S / B / vlo of the listed reads (20 B) + their list
        # entries (8 B out); K2b: difference array in (4 B) and summary + flag out (17 B) per window, list entries in (8 B),
        # haplotype-0 record (32 B) per interesting window, 20 B per extra key
        "k2_ms": n_reads * 10 + n_special * (20 + 8 + 8) + n_win * (4 + 4 + 17) + (t_res["n_interesting"] + n_records) * 32 + n_records * 2 * 20 + n_seg * (96 + 16) + n_chunk * 32,
        "k3_ms": n_records * 2 * (16 + 4 + 32) + view.ref_bytes + n_seg * 96 + n_chunk * 32,
        "k4_ms": n_win * 2 + t_res["n_interesting"] * (4 + 2 * 48),
        "k5_ms": n_win * 3 + n_records * (64 + 64 + 48 + 32),
    }
    # k_replay (irregular transcripts) is a latency-bound dependent chain, not a streaming kernel: it counts in ms_per_step
    # but is not a roofline candidate
    dom = max(alg, key=lambda k: per_kernel[k])
    dom_ms = per_kernel[dom] / args.steps
    achieved = alg[dom] / (dom_ms / 1000.0) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get(name, {}).get(dom)  # per workload: DRAM bytes of one launch from the committed ncu capture
    roofline = {"bound": "hbm", "kernel": {"k1_ms": "k_allele_call", "k2_ms": "k_read_runs + k_window_hist", "k3_ms": "k_assemble", "k4_ms": "compaction",
                                           "k5_ms": "record kernels"}[dom],
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "timed": "every kernel alone on one stream (MPH_SIDE_REPLAY=0), %d steps after the timed loop" % args.steps,
                "kernel_ms": {k: v / args.steps for k, v in per_kernel.items()},
                "kernel_ms_in_timed_loop": {k: v / args.steps for k, v in per_kernel_overlapped.items()},
                "serial_chain_ms": serial_chain_ms / args.steps,
                "pipeline_GBs": sum(alg.values()) / (dev_ms / 1000.0) / 1e9, "pipeline_frac": sum(alg.values()) / (dev_ms / 1000.0) / 1e9 / peak,
                # SURVEY.md §8(d) models 550 B per window (every read ships its packed bases); this design ships far less
                # (DESIGN.md §5), so that figure over this run time overstates the bandwidth actually moved - reported for reference
                "survey_model": {"bytes_per_window": 550, "GBs": 550.0 * n_win / (dev_ms / 1000.0) / 1e9,
                                 "frac": 550.0 * n_win / (dev_ms / 1000.0) / 1e9 / peak}}

    # ---- CPU baseline, parity of the benched batch, files -> files: one oracle run on a bounded slice of the rank-0 shard
    cpu, parity_checked, e2e_files = None, 0, None
    if not args.no_cpu_baseline:
        ensure_oracle()
        with tempfile.TemporaryDirectory() as tmp:
            sample_tx = min(w["n_transcripts"], args.cpu_sample_transcripts)
            d = os.path.join(tmp, "sample")
            write_sample_files(name, sample_tx, shard_seed(0), d)
            p, stats = run_oracle(d, "one", mode)
            t_o = time.perf_counter()
            p.wait()
            oracle_wall = time.perf_counter() - t_o
            st = json.load(open(stats))
            cpu = {"value": st["windows"] / st["phase_s"], "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": "first %d of %d transcripts of the rank-0 shard (the same genes, reads and variants as the packed batch): %d windows, %d read*windows in %.1f s (BAM decode included)" %
                             (sample_tx, w["n_transcripts"], st["windows"], st["read_windows"], st["phase_s"]),
                   "read_windows_per_s": st["read_windows"] / st["phase_s"]}
            streams = [("fa", "out.fa"), ("tsv", "out.tsv")] + ([("n.fa", "out.normal.fa")] if mode == "somatic" else [])
            # (1) the benched batch: the oracle's bytes must be a prefix of what the GPU result writes (records of the first
            #     transcripts do not depend on the later ones)
            outs = {n: os.path.join(tmp, "gpu_" + n) for _, n in streams}
            last.write(outs["out.fa"], outs["out.tsv"], outs.get("out.normal.fa", os.path.join(tmp, "gpu_unused")))
            for ext, n in streams:
                want = open(os.path.join(d, "o_one." + ext), "rb").read()
                got = open(outs[n], "rb").read(len(want))
                if got != want:
                    raise SystemExit("PARITY FAILURE: %s of the benched batch differs from the oracle on its first %d transcripts" % (n, sample_tx))
                if n == "out.tsv":
                    parity_checked = max(0, want.count(b"\n") - 1)
            # (2) files -> files through the file driver on the same slice
            fo = {n: os.path.join(tmp, "files_" + n) for _, n in streams}
            runs = []
            for rep in range(3):
                t_f = time.perf_counter()
                if mode == "normal":
                    ctx.run_normal(os.path.join(d, "reads.bam"), os.path.join(d, "ref.fa"), os.path.join(d, "variants.vcf"), os.path.join(d, "annotation.gtf"),
                                   fo["out.fa"], fo["out.tsv"])
                else:
                    ctx.run_somatic(os.path.join(d, "reads.bam"), os.path.join(d, "ref.fa"), os.path.join(d, "variants.vcf"), os.path.join(d, "annotation.gtf"),
                                    fo["out.fa"], fo["out.tsv"], fo["out.normal.fa"])
                runs.append((time.perf_counter() - t_f, ctx.timing()))
            for ext, n in streams:
                if open(fo[n], "rb").read() != open(os.path.join(d, "o_one." + ext), "rb").read():
                    raise SystemExit("PARITY FAILURE: %s of the file driver differs from the oracle" % n)
            wall_f, t_f = min(runs, key=lambda x: x[0])
            cores = os.cpu_count() or 1
            e2e_files = {"value": st["windows"] / wall_f, "unit": UNIT, "seconds": wall_f, "transcripts": sample_tx, "windows": st["windows"],
                         "stages_ms": {k: t_f[k] for k in ("ingest_ms", "pack_ms", "h2d_ms", "d2h_ms", "residue_ms", "write_ms", "total_ms")},
                         "oracle_1core": {"value": st["windows"] / oracle_wall, "seconds": oracle_wall},
                         "oracle_all_cores_estimate": {"value": st["windows"] / oracle_wall * cores, "cores": cores,
                                                       "note": "the reference is single-threaded per invocation; independent processes on disjoint gene ranges scale with the cores (--impl reference measures it)"},
                         "ratio_vs_oracle_1core": oracle_wall / wall_f, "ratio_vs_oracle_all_cores_estimate": oracle_wall / wall_f / cores,
                         "outputs_identical_to_oracle": True}
    last.close()

    line = {
        "metric": METRIC, "value": windows_all / (dev_ms_max / 1000.0), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms_max, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": config_of(name),
        "shape": {"windows_per_gpu": windows, "reads_per_gpu": n_reads, "read_windows_per_gpu": read_windows, "records_per_gpu": n_records,
                  "host_residue_windows_per_gpu": t_res["n_interesting"], "replay_units_per_gpu": t_res["n_replay_units"],
                  "h2d_GB_per_gpu": view.h2d_bytes / 1e9, "generation_and_packing_s": gen_s},
        "read_windows_per_s": rw_all / (dev_ms_max / 1000.0),
        "e2e": {"value": windows_all / (e2e_ms_max / 1000.0), "unit": UNIT, "h2d_bytes_per_step": h2d_b, "d2h_bytes_per_step": d2h_b,
                "ms_per_step": e2e_ms_max, "calls_timed": n_e2e, "stages_ms": stage},
        "e2e_files": e2e_files,
        "parity_checked": parity_checked,
        "gpu_launches": launches_timed,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "clocks": summarize_clocks(clk_lines),
        "wall_s_resident_loop": wall_res,
    }
    print(json.dumps(line))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
