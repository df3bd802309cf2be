#!/usr/bin/env python
"""bench.py -- the k-mer hot path on B200, one JSON line per run.

Workload (BASELINE.json configs[3], the one the metric is quoted on): one synthetic
3.1 Gbp sequence (seeded generator of include/dnagpu_synth.h, every 8th 1024-base block a
planted repeat), k = 31, `GROUP BY kmer` with total / distinct / unique.  Total work is fixed,
so scaling is "strong".

N > 1 (one process per GPU, torch.distributed / NCCL for the plumbing), `--exchange`:
  gather (default)  the sequence stays sharded by base range, one shard per GPU with its (k-1)-base
          overlap, every shard mapped into every GPU's address space (CUDA IPC peer memory); each GPU
          walks ALL shards over NVLink and counts the k-mers dnagpu_owner_of assigns to it.  What
          crosses NVLink is the 2-bit packed bases, not 8-byte k-mers; the only collective is the
          final all-reduce of the three aggregates.
  peer / fused / routed   k-mers routed to their owners (scatter kernel storing into peer memory /
          NCCL all-to-all); kept for comparison and used by the reads workload (WHERE clause).

  value   Gkmer/s with the packed words already resident in HBM (every kernel of the query:
          extract + partition + count + aggregates), CUDA-event timed, max over ranks.
  e2e     the same query from HOST buffers: pinned host words -> H2D -> count -> D2H of the three
          aggregates, every step.  N = 1: the C-ABI call dnagpu_count_kmers().  N > 1: every rank
          uploads its shard, then the same count.
  roofline  the kernel with the largest share of the step (CUDA events around every launch, taken
          inside the timed region): its algorithmic bytes / its average duration, plus the same
          figure for every kernel of the pipeline and for the whole step.  Kernels that read
          0.25 B/base and test every position (the fused WHERE scan) carry "bound": "issue" and are
          measured against the instruction-issue peak instead.
  cpu_baseline  the reference's own dna.c (oracle/_ref: compiled unmodified against a PostgreSQL
          API shim and driven like the executor) on the host cores, bounded sample, all threads;
          cpu_baseline_1thread is the same on ONE thread, which is how PostgreSQL runs this plan
          (generate_kmers is not PARALLEL SAFE).

Other workloads: --workload c1 (10 kb, k = 5: BASELINE configs[0], the CPU reference timed in full),
c2 (100 Mbp, k = 21), c3 (100 M reads, fused WHERE + count), c5 (k = 3..32 sweep over 1 Gbp, one line).
Every result is compared with the CPU oracle's answer for the exact workload
(tests/golden/big_expected.json); a run that differs prints no line.

`--impl reference` times the reference's CPU implementation of the same query
(oracle/_ref = the reference's own dna.c when it could be compiled, else the oracle port).

`--dump-outputs DIR` writes what the timed legs returned in their last step as DIR/<name>.npy (float64), so that
two builds can be compared output for output (the inputs are generated from fixed seeds):
  stats         total, distinct, unique of the resident-input leg (c5: one row k, total, distinct, unique per k)
  stats_e2e     the same from the host-buffer leg
  extract_rows  a fixed, seeded sample of the extraction leg's rows: row index, high and low 32 bits of the k-mer
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "dna-sequences-pg-extension_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

WORKLOADS = {
    # name: (n_bases, k, seed, description)      -- BASELINE.json configs[3], [1], [4], [0]
    "c4": (3_100_000_000, 31, 4, "3.1 Gbp synthetic sequence, k=31 GROUP BY kmer count + total/distinct/unique"),
    "c2": (100_000_000, 21, 2, "100 Mbp synthetic sequence, k=21 full count + total/distinct/unique"),
    "c5": (1_000_000_000, 31, 5, "k-sweep 3..32 over a 1 Gbp synthetic sequence (dense tables, partition path, "
                                 "k=32 full-uint64 sentinel)"),
    "c1": (10_000, 5, 1, "generate_kmers + GROUP BY count, k=5, one 10 kb synthetic sequence"),
    # BASELINE.json configs[2]: reads (each its own dna value), WHERE ^@ AND @> fused into the count
    "c3": (100_000_000 * 150, 31, 3, "100M synthetic 150 bp reads, k=31, WHERE kmer ^@ 'AC' AND "
                                     "'NNNNNNNNNNNNWSNNNNNNNNNNNNNNNRY' @> kmer, fused filter-count"),
}
READS = {"c3": {"n_reads": 100_000_000, "bases": 150, "stride": 5, "prefix": "AC",
                "pattern": "NNNNNNNNNNNNWSNNNNNNNNNNNNNNNRY"}}
REPEAT_EVERY = 8
METRIC = "Gkmer/s counted (k=31) at 1/2/4/8 B200; extraction HBM GB/s vs peak"
NVLINK_PEER_GBS = 770.0   # measured peer-copy rate per direction per GPU (B200_PROFILING.md)
SM_COUNT, LANES_PER_SM = 148, 128


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


DUMP_ROWS = 1 << 20  # rows of the extraction leg sampled by --dump-outputs (at most 24 MB as float64)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: one DIR/<name>.npy per array, as float64 (every value dumped is below 2**53, so exact)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def golden(name):
    try:
        with open(os.path.join(ROOT, "tests", "golden", "big_expected.json")) as f:
            return json.load(f).get(name)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ============================== the reference arm ==============================
CHUNK_BASES = 1 << 16  # the CPU arms cut the sample into overlapping chunks, one dna value each


def cpu_reference_rate(n_bases, k, seed, threads, sample_bases, reads=None):
    """Time the reference's CPU implementation of the query on a prefix of the workload.

    oracle/_ref (the reference's own dna.c, compiled unmodified against the PostgreSQL API shim and
    driven like the executor: SRF loop + HashAggregate through kmer_hash/kmer_eq) when it is built,
    else the oracle's faithful restatement.  The prefix is cut into chunks of 65536 start positions
    (each chunk a dna value overlapping the next by k-1 bases, so every k-mer is produced once) so
    that all host threads have work; PostgreSQL itself would run the plan on ONE core because
    generate_kmers is not PARALLEL SAFE (dna--1.0.sql:188-191).  A workload no longer than one chunk
    (c1) is run whole, as one dna value.
    Returns (Gkmer/s, seconds, (total, distinct, unique), kind, bases)."""
    from oracle import ref_cpu as R
    from oracle import ref_real as P
    kind = "reference" if os.path.exists(P.SO) else "port"
    if reads is not None:  # a prefix of the batch of reads, each read one dna value
        n = max(threads, sample_bases // reads["bases"])
        words = R.synth_reads(seed, n, reads["bases"], reads["stride"], REPEAT_EVERY)
        pk = R.kmer_make(reads["prefix"])
        t0 = time.perf_counter()
        if kind == "reference":
            r = P.count(words, n, reads["bases"], reads["stride"], k, prefix=pk, pattern=reads["pattern"],
                        threads=threads, want_rows=False)
        else:
            r = R.count_query(words, n, reads["bases"], reads["stride"], k, prefix=pk, pattern=reads["pattern"],
                              faithful=True, threads=threads, want_rows=False)
        dt = time.perf_counter() - t0
        rows = n * (reads["bases"] - k + 1)  # k-mers generated and tested, the unit of the metric
        return rows / dt / 1e9, dt, (rows,) + tuple(r.stats[1:]), kind, n * reads["bases"]
    if n_bases <= CHUNK_BASES:
        import numpy as np
        words = np.concatenate([R.synth_seq(seed, n_bases, REPEAT_EVERY), np.zeros(1, dtype=np.uint64)])
        t0 = time.perf_counter()
        if kind == "reference":
            r = P.count(words, 1, n_bases, words.size, k, threads=1, want_rows=False)
        else:
            r = R.count_query(words, 1, n_bases, words.size, k, faithful=True, threads=1, want_rows=False)
        dt = time.perf_counter() - t0
        return r.total / dt / 1e9, dt, r.stats, kind, n_bases
    n_chunks = max(1, (sample_bases - (k - 1)) // CHUNK_BASES)
    sample = n_chunks * CHUNK_BASES + k - 1
    words = R.synth_seq(seed, n_bases, REPEAT_EVERY, first_word=0, n_words=(sample + 31) // 32 + 1)
    t0 = time.perf_counter()
    if kind == "reference":
        r = P.count(words, n_chunks, CHUNK_BASES + k - 1, CHUNK_BASES // 32, k, threads=threads, want_rows=False)
    else:
        r = R.count_query(words, n_chunks, CHUNK_BASES + k - 1, CHUNK_BASES // 32, k, faithful=True,
                          threads=threads, want_rows=False, expected_keys=sample)
    dt = time.perf_counter() - t0
    assert r.total == n_chunks * CHUNK_BASES
    return r.total / dt / 1e9, dt, r.stats, kind, sample


REF_WHAT = {"reference": "the reference's own dna.c (unmodified, PostgreSQL API shim) driven like the executor: "
                         "generate_kmers SRF loop + hash aggregate through kmer_hash/kmer_eq",
            "port": "oracle port: faithful per-k-mer decode/validate/encode of dna.c:803-825 + kmer_hash/kmer_eq "
                    "hash aggregate"}


def cpu_baselines(n_bases, k, seed, reads, sample, sample_1t):
    """(all-threads baseline, one-thread baseline) objects for the JSON line."""
    threads = max(1, min(os.cpu_count() or 1, 64))
    cv, cdt, _, ckind, csample = cpu_reference_rate(n_bases, k, seed, threads, sample, reads)
    cpu = {"value": cv, "unit": "Gkmer/s", "cores": threads if csample > CHUNK_BASES or reads else 1, "kind": ckind,
           "sample": f"first {csample} bases of the workload ({cdt:.1f} s), {REF_WHAT[ckind]}"
                     + ("" if csample < n_bases else " -- the whole workload")}
    ov, odt, _, okind, osample = cpu_reference_rate(n_bases, k, seed, 1, sample_1t, reads)
    one = {"value": ov, "unit": "Gkmer/s", "cores": 1, "kind": okind,
           "sample": f"first {osample} bases of the workload ({odt:.1f} s) on ONE thread -- how PostgreSQL runs this "
                     "plan: generate_kmers / ^@ / @> are not PARALLEL SAFE (dna--1.0.sql:188-201, 268-276)"}
    return cpu, one


def run_reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return 0
    n_bases, k, seed, desc = WORKLOADS[args.workload]
    k = args.k or k
    threads = max(1, min(os.cpu_count() or 1, 64))
    reads = READS.get(args.workload)
    if args.cpu_large_sample:
        sample = args.cpu_large_sample
    else:
        # calibrate the per-step sample so that the whole run ends within a few minutes
        rate, dt, _, kind, _ = cpu_reference_rate(n_bases, k, seed, threads, 4_000_000, reads)
        # the rate on a small (cache-friendly) sample is optimistic: keep 40 % of the time budget
        budget_s = 0.4 * max(0.5, min(4.0, 100.0 / max(1, args.steps + args.warmup)))
        sample = int(max(1_000_000, min(16_000_000, rate * 1e9 * budget_s)))
    for _ in range(args.warmup):
        cpu_reference_rate(n_bases, k, seed, threads, sample, reads)
    wall, total = 0.0, 0
    for _ in range(args.steps):
        _, dt, stats, kind, sample_used = cpu_reference_rate(n_bases, k, seed, threads, sample, reads)
        wall += dt
        total += stats[0]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"stats": stats})
    value = total / wall / 1e9
    sample_desc = (f"first {sample_used} bases of the workload per step, {REF_WHAT[kind]}, {threads} threads "
                   "(Postgres itself would run this serially: generate_kmers is PARALLEL UNSAFE; the hash table of a "
                   "sample this small is cache-resident, which flatters the CPU side)")
    ov, odt, _, okind, osample = cpu_reference_rate(n_bases, k, seed, 1, min(sample, 1_000_000), reads)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Gkmer/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(1, args.steps),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": desc, "n_bases": n_bases, "k": k, "seed": seed, "repeat_every": REPEAT_EVERY,
                   "sample_bases_per_step": sample_used},
        "cpu_baseline": {"value": value, "unit": "Gkmer/s", "cores": threads, "kind": kind, "sample": sample_desc},
        "cpu_baseline_1thread": {"value": ov, "unit": "Gkmer/s", "cores": 1, "kind": okind,
                                 "sample": f"first {osample} bases ({odt:.1f} s), one thread"},
        "e2e": {"value": value, "unit": "Gkmer/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ================================= our arm =====================================
# Executed SASS instructions per start position of the kernels that read 0.25 B/base and test EVERY position (issue-bound,
# not HBM-bound).  Defaults: the plane test from an ncu capture (profiles/r02c_c3_filter_planes_summary.csv: 7.34e8 warp
# instructions for 1.2e9 positions = 19.6), the Shift-And scan and the ownership scan from their SASS listings
# (profiles/r02_sass_hot_kernels.txt); profiles/issue.json overrides them with ncu counts of the current build.
# Integer SASS runs on two pipes of HALF the issue rate each (ALU: LOP3 / SHF / IADD3 / ISETP, FMA: IMAD): a kernel that is
# mostly ALU-pipe instructions saturates at frac ~ 0.5 of the issue peak.
ISSUE_INSTR_PER_POSITION = {"filter_collect": 9.5, "filter_count": 9.5, "filter_collect:planes": 19.6, "collect_owned": 27.4,
                            "collect_owned:2": 30.75, "collect_owned:4": 19.39, "collect_owned:8": 11.72}


def issue_table():
    try:
        with open(os.path.join(ROOT, "profiles", "issue.json")) as f:
            t = dict(ISSUE_INSTR_PER_POSITION)
            t.update({k_: float(v) for k_, v in json.load(f).items() if not k_.startswith("_")})
            return t
    except Exception:
        return dict(ISSUE_INSTR_PER_POSITION)


def run_sweep(args, ctx, torch, dev, stream, peak, peak_src):
    """--workload c5: GROUP BY kmer for every k from 3 to 32 over the 1 Gbp sequence, method AUTO.  One line:
    per-k time, method and result, each checked against the oracle; value = all k-mers of the sweep / its time."""
    n_bases, _, seed, desc = WORKLOADS["c5"]
    n_bases = args.n_bases or n_bases
    seq = ctx.synth(n_bases, seed, REPEAT_EVERY)
    host = torch.empty(seq.n_words + 2, dtype=torch.int64, pin_memory=True)
    host.zero_()
    assert ctx.lib.dnagpu_seq_download(ctx.handle, seq.handle, C.c_void_p(host.data_ptr()), seq.n_words) == 0
    ks = list(range(3, 33))
    per_k, total_rows, total_ms, launches = {}, 0, 0.0, 0
    dumped = {"stats": [], "stats_e2e": []}
    sampler = ClockSampler(dev.index)
    sampler.start()
    for k in ks:
        for _ in range(max(1, min(args.warmup, 3))):
            st, _ = ctx.count(seq, k)
        ctx.profile(True)
        ctx.profile_reset()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record(stream)
        for _ in range(args.steps):
            st, _ = ctx.count(seq, k)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        kernels = ctx.profile_dump()
        ctx.profile(False)
        ms = e0.elapsed_time(e1) / args.steps
        g = golden(f"c5_k{k}") if not args.n_bases else None
        res = (st.total, st.distinct, st.unique)
        dumped["stats"].append((k,) + res)
        if g is not None and res != (g["total"], g["distinct"], g["unique"]):
            print(f"bench: k={k}: result {res} differs from the oracle's {(g['total'], g['distinct'], g['unique'])}: "
                  "no line printed", file=sys.stderr)
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, {"stats": dumped["stats"]})
            return 1
        method = ("dense" if any(n.startswith("count_dense") for n in kernels) else
                  "partition" if "count_buckets" in kernels else "hash")
        per_k[str(k)] = {"ms": ms, "gkmer_s": st.total / ms / 1e6, "method": method, "distinct": st.distinct,
                         "unique": st.unique, "oracle": "equal" if g is not None else "not compared"}
        total_rows += st.total
        total_ms += ms
        launches += sum(v["launches"] for v in kernels.values())
    clocks = sampler.stop()
    t0 = time.perf_counter()
    for k in ks:  # the host-buffer call for every k: 250 MB H2D each
        st = ctx.count_kmers_ptr(C.c_void_p(host.data_ptr()), n_bases, k)
        dumped["stats_e2e"].append((k, st.total, st.distinct, st.unique))
    e2e_s = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dumped)
    slow = max(per_k, key=lambda q: per_k[q]["ms"])
    cpu, one = cpu_baselines(n_bases, 31, seed, None, args.cpu_sample, 1_000_000)
    # roofline of the slowest k: the partition pipeline moves 0.25 B/base + 8 + 16 + 8 B per k-mer (DESIGN.md 4)
    pipe_bytes = 0.25 * n_bases + 32.0 * per_k[slow]["gkmer_s"] * per_k[slow]["ms"] * 1e6
    line = {
        "metric": METRIC, "value": total_rows / total_ms / 1e6, "unit": "Gkmer/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": desc, "n_bases": n_bases, "k": "3..32", "seed": seed, "repeat_every": REPEAT_EVERY,
                   "unit_of_value": "k-mers counted per second over the 30 runs of the sweep (a step = all 30)",
                   "l2": "inputs larger than L2 for k >= 13; k <= 12 tables are L2-resident by design"},
        "per_k": per_k,
        "result": {"oracle": "every k equal to tests/golden/big_expected.json" if not args.n_bases else "not compared"},
        "e2e": {"value": total_rows / e2e_s / 1e9, "unit": "Gkmer/s", "ms_per_step": 1e3 * e2e_s,
                "h2d_bytes_per_step": int(8 * ((n_bases + 31) // 32)) * len(ks), "d2h_bytes_per_step": 24 * len(ks),
                "api": "dnagpu_count_kmers(ctx, host_words, n_bases, k, NULL, &stats, NULL) for k = 3..32"},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "kernel": f"whole count pipeline at k={slow} (the slowest k)",
                     "achieved": pipe_bytes / per_k[slow]["ms"] / 1e6, "peak": peak, "unit": "GB/s",
                     "frac": pipe_bytes / per_k[slow]["ms"] / 1e6 / peak, "traffic": None, "peak_source": peak_src},
        "cpu_baseline": cpu, "cpu_baseline_1thread": one, "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    seq.free()
    return 0


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import dnagpu
    from dnagpu.distributed import (GpuEngine, PeerExchange, ShardRing, count_sharded, count_sharded_fused,
                                    count_sharded_gather, count_sharded_peer, reads_shard_of, shard_of)

    rank, world, local = dist_env()
    n_bases, k, seed, desc = WORKLOADS[args.workload]
    k = args.k or k
    reads = READS.get(args.workload)
    if args.n_bases:
        n_bases = args.n_bases
        if reads:
            reads = dict(reads, n_reads=max(world, n_bases // reads["bases"]))
            n_bases = reads["n_reads"] * reads["bases"]
    where = {"prefix": reads["prefix"], "pattern": reads["pattern"]} if reads else {}
    if reads and args.planes:
        where["planes"] = True  # A/B: the per-position plane test instead of the Shift-And automaton (single GPU)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(device=dev)
    peak, peak_src = measured_peaks()
    if reads and args.exchange == "gather":
        args.exchange = "peer"  # a WHERE clause: the rows that pass are routed (few), not the bases
    gather = world > 1 and args.exchange == "gather"

    with torch.cuda.stream(stream):
        ctx = dnagpu.Context(local, torch_stream=True)
        if args.workload == "c5" and not args.k:
            if world > 1:
                if rank == 0:
                    print("bench: the k-sweep workload is a single-GPU line", file=sys.stderr)
                return 2
            return run_sweep(args, ctx, torch, dev, stream, peak, peak_src)
        ring = None
        if reads:
            first, starts = reads_shard_of(reads["n_reads"], world, rank)  # first read, reads of this rank
            seq = ctx.synth_reads(first, starts, reads["bases"], reads["stride"], seed, REPEAT_EVERY)
            n_rows_total = reads["n_reads"] * (reads["bases"] - k + 1)
        elif gather:
            ring = ShardRing(ctx, world, rank, n_bases)  # collective
            first, starts = ring.my_shard
            seq = ctx.synth_range(n_bases, seed, REPEAT_EVERY, first, starts, 32)
            n_rows_total = n_bases - k + 1
        else:
            first, starts = shard_of(n_bases, k, world, rank)
            seq = ctx.synth_range(n_bases, seed, REPEAT_EVERY, first, starts, k)
            n_rows_total = n_bases - k + 1
        n_words_local = seq.n_words
        n_words_total = (n_bases + 31) // 32 if not reads else reads["n_reads"] * reads["stride"]
        # host copy of this rank's packed words, pinned (the dna value a backend would hold)
        host = torch.empty(n_words_local + 2, dtype=torch.int64, pin_memory=True)
        host.zero_()
        ctx.synchronize()
        rc = ctx.lib.dnagpu_seq_download(ctx.handle, seq.handle, C.c_void_p(host.data_ptr()), n_words_local)
        assert rc == 0
        local_bases = starts * reads["bases"] if reads else min(n_bases - first, starts + k - 1)
        if gather:
            ctx.fill_words(ring.local, seq, ring.n_words[rank])
            ring.publish()

        def barrier():
            if world > 1:
                dist.barrier(device_ids=[local])
            torch.cuda.synchronize(dev)

        engine = GpuEngine(ctx) if world > 1 else None
        xbuf = {}
        px = None
        if world > 1 and args.exchange == "peer":
            try:  # collective: raises on every rank or on none
                px = PeerExchange(ctx, world, rank, int(n_rows_total / world * 1.15) + (1 << 20))
            except RuntimeError as e:
                if rank == 0:
                    print(f"bench: {e}; falling back to --exchange fused", file=sys.stderr)
                args.exchange = "fused"

        def count_resident(s):
            """One pass of the hot path with the packed words resident in HBM -> (total, distinct, unique)."""
            if world == 1:
                st, _ = ctx.count(s, k, table=False, load_factor=args.load_factor, **where)
                return st.total, st.distinct, st.unique
            if gather:
                return count_sharded_gather(ctx, ring, k)
            if args.exchange == "peer":
                return count_sharded_peer(ctx, s, k, n_rows_total, world, rank, px, **where)
            if args.exchange == "fused":
                return count_sharded_fused(ctx, s, k, n_rows_total, world, rank, xbuf, chunks=args.chunks, **where)
            return count_sharded(engine, s, k, world, load_factor=args.load_factor, **where)

        def count_e2e():
            """Host words in, aggregates out (H2D and D2H inside)."""
            hp = C.c_void_p(host.data_ptr())
            if world == 1 and reads:
                st = ctx.count_reads_ptr(hp, starts, reads["bases"], reads["stride"], k, **where)
                return st.total, st.distinct, st.unique
            if world == 1:
                st = ctx.count_kmers_ptr(hp, local_bases, k)
                return st.total, st.distinct, st.unique
            if gather:  # this rank's shard: pinned host -> its ring buffer; then everybody reads everybody's
                ctx.upload_to(ring.local, host[:n_words_local], ring.n_words[rank])
                ring.publish()
                return count_sharded_gather(ctx, ring, k)
            if reads:
                s = ctx.upload_reads_ptr(hp, starts, reads["bases"], reads["stride"])
            else:
                s = ctx.upload_words(hp, local_bases)
                s.set_start_limit(starts)
            r = count_resident(s)
            s.free()
            return r

        # ---- value leg: resident inputs, CUDA events ----
        for _ in range(args.warmup):
            stats = count_resident(seq)
        ctx.profile(True)
        ctx.profile_reset()
        sampler = ClockSampler(local)
        barrier()
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            stats = count_resident(seq)
        e1.record(stream)
        barrier()
        clocks = sampler.stop() if rank == 0 else None
        ms = e0.elapsed_time(e1)
        kernels = ctx.profile_dump()
        ctx.profile(False)
        ctx.profile_reset()

        # ---- e2e leg: host buffers in, aggregates out, wall clock around synchronous calls ----
        # Gather form: two shard rings; the H2D of step s + 1 (copy stream) runs under the count of step s.  Every step
        # still uploads its own input and reads its own result inside the timed region.
        ring2, copy_stream = None, None
        if gather:
            try:  # collective: raises on every rank or on none
                ring2 = ShardRing(ctx, world, rank, n_bases)
                copy_stream = torch.cuda.Stream(device=dev)
            except RuntimeError as e:
                if rank == 0:
                    print(f"bench: no second shard ring ({e}); the e2e uploads are not overlapped", file=sys.stderr)

        def e2e_steps(n_steps):
            if ring2 is None:
                r = None
                for _ in range(n_steps):
                    r = count_e2e()
                return r
            rings, r = [ring, ring2], None

            def upload(rg):
                copy_stream.wait_stream(stream)  # nothing of ours still reads that ring (the all-reduce fenced the peers)
                with torch.cuda.stream(copy_stream):
                    ctx.upload_to(rg.local, host[:n_words_local], rg.n_words[rank])
            upload(rings[0])
            for s_ in range(n_steps):
                copy_stream.synchronize()          # this rank's shard of step s_ is in place ...
                dist.barrier(device_ids=[local])   # ... and everybody's
                if s_ + 1 < n_steps:
                    upload(rings[(s_ + 1) % 2])
                r = count_sharded_gather(ctx, rings[s_ % 2], k)
            return r

        e2e_steps(min(args.warmup, 2))
        barrier()
        t0 = time.perf_counter()
        stats_e2e = e2e_steps(args.e2e_steps)
        barrier()
        e2e_s = time.perf_counter() - t0
        e2e_overlapped = ring2 is not None
        if ring2 is not None:
            ring2.close()

        # ---- extraction GB/s (the second half of the metric), timed on its own ----
        extract, extract_rows = None, None
        if not args.no_extract and not reads and n_bases >= 1_000_000:
            xs_bases = min(local_bases, 1_000_000_000)
            xs = ctx.synth_range(n_bases, seed, REPEAT_EVERY, first, max(0, xs_bases - k + 1), k)
            xr = xs.kmer_count(k)
            xout = torch.empty(xr + 2, dtype=torch.int64, device=dev)
            for _ in range(3):
                ctx.extract(xs, k, out=xout)
            x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            x0.record(stream)
            xn = args.steps
            for _ in range(xn):
                ctx.extract(xs, k, out=xout)
            x1.record(stream)
            torch.cuda.synchronize(dev)
            xms = x0.elapsed_time(x1) / xn
            if args.dump_outputs:
                idx = np.unique(np.random.default_rng(0).integers(0, xr, size=min(xr, DUMP_ROWS)))
                rows = xout[torch.from_numpy(idx).to(dev)].cpu().numpy().view(np.uint64)
                extract_rows = np.stack([idx, rows >> 32, rows & 0xFFFFFFFF], axis=1)
            xbytes = 0.25 * xs_bases + 8.0 * xr
            extract = {"rows": xr, "ms": xms, "gkmer_s": xr / xms / 1e6, "gbs": xbytes / xms / 1e6,
                       "frac": xbytes / xms / 1e6 / peak, "bytes_per_row": 8.25,
                       "note": f"output (8 B/row) larger than L2; {xn} back-to-back launches"}
            # ... and the WHERE clause over those materialised rows (kmer ^@ 'AC': 1/16 of them pass), rows kept in order
            from dnagpu import _where
            fw, _keep = _where("AC", None)
            fres = torch.empty(xr // 8 + 2, dtype=torch.int64, device=dev)
            fn = C.c_uint64()

            def scan():
                rc_ = ctx.lib.dnagpu_filter_keys(ctx.handle, xout.data_ptr(), xr, k, C.byref(fw), fres.data_ptr(),
                                                 fres.numel(), C.byref(fn))
                assert rc_ == 0, rc_
            for _ in range(2):
                scan()
            torch.cuda.synchronize(dev)
            x0.record(stream)
            for _ in range(xn):
                scan()
            x1.record(stream)
            torch.cuda.synchronize(dev)
            fms = x0.elapsed_time(x1) / xn
            fbytes = 2 * 8.0 * xr + 8.0 * fn.value  # the column is read twice (count per tile, ordered write)
            extract["filter_keys"] = {"predicate": "kmer ^@ 'AC'", "rows": xr, "matches": int(fn.value), "ms": fms,
                                      "gkmer_s": xr / fms / 1e6, "gbs": fbytes / fms / 1e6,
                                      "frac": fbytes / fms / 1e6 / peak,
                                      "note": "bytes = 2 passes over the 8 B rows + rows written"}
            del xout, fres
            xs.free()

    # ---- reduce over ranks ----
    if world > 1:
        t = torch.tensor([ms, e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s = t.tolist()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"stats": stats, "stats_e2e": stats_e2e,
                                         **({"extract_rows": extract_rows} if extract_rows is not None else {})})
    assert reads or stats[0] == n_rows_total, (stats, n_rows_total)
    assert tuple(stats) == tuple(stats_e2e), (stats, stats_e2e)
    # parity gate: the CPU oracle's answer for this exact workload (tests/golden/big_expected.json, produced by
    # tests/golden/make_golden_big.py).  A run whose result differs prints NO line.
    gold = None
    if not args.n_bases:
        gold = golden({"c4": "c4", "c2": "c2", "c5": f"c5_k{k}", "c3": "c3", "c1": "c1"}[args.workload])
        if gold is not None and gold.get("k") != k:
            gold = None
        if gold is not None and tuple(stats) != (gold["total"], gold["distinct"], gold["unique"]):
            if rank == 0:
                print(f"bench: result {tuple(stats)} differs from the oracle's "
                      f"{(gold['total'], gold['distinct'], gold['unique'])}: no line printed", file=sys.stderr)
            return 1

    if rank == 0:
        value = n_rows_total * args.steps / (ms * 1e-3) / 1e9
        e2e_value = n_rows_total * args.e2e_steps / e2e_s / 1e9
        launches = sum(v["launches"] for v in kernels.values())
        # algorithmic bytes per launch of every kernel of the count pipeline (DESIGN.md section 4):
        # rows = k-mers one launch handles on this rank; base reads are 0.25 B/base
        rows_r = stats[0] / world          # keys that reach the partition / count stages (after WHERE)
        rows_tested_r = n_rows_total / world   # start positions one rank's predicate scan tests
        base_b = 8.0 * n_words_local       # the packed words one launch reads (0.25 B/base)
        listed = "filter_collect" in kernels and kernels["filter_collect"]["launches"] > 0
        l1_from_list = listed or gather    # level 1 reads a key list (8 B/key) instead of packed words
        ALG = {
            "count_hash": base_b + 16.0 * rows_r, "count_hash_keys": 8.0 * rows_r + 16.0 * rows_r,
            "count_dense": base_b + 4.0 * rows_r, "count_dense_smem": base_b,
            # exact level 1 (N > 1 routed forms, WHERE clause): histogram over the packed words or the key list
            "part_hist": 8.0 * rows_r if listed else base_b,
            "part_scatter": (8.0 * rows_r if l1_from_list else base_b) + 8.0 * rows_r,
            # level 1 fused with the exchange: packed words in, 8 B per k-mer out (local or over NVLink)
            "part_scatter_peer": (8.0 * rows_r if listed else base_b) + 8.0 * rows_r,
            # gather form: EVERY base of the sequence is read (all shards), the owned k-mers are written
            "collect_owned": 8.0 * n_words_total + 8.0 * rows_r,
            # a WHERE clause is evaluated once into a key list: packed words in, matching rows out
            "filter_collect": base_b + 8.0 * rows_r,
            "part_hist2": 8.0 * rows_r, "part_scatter2": 16.0 * rows_r, "count_buckets": 8.0 * rows_r,
            "partition_count": base_b, "partition_write": base_b + 8.0 * rows_r,
        }
        issue = issue_table()
        if args.planes:
            issue["filter_collect"] = issue["filter_collect:planes"]
        if f"collect_owned:{world}" in issue:  # the ownership scan costs less per position for 2 / 4 / 8 owners (linear form)
            issue["collect_owned"] = issue[f"collect_owned:{world}"]
        issue = {q: v for q, v in issue.items() if ":" not in q}
        clk_hz = 1e6 * float((clocks or {}).get("sm_mhz") or 1965.0)
        issue_peak = SM_COUNT * LANES_PER_SM * clk_hz / 1e12  # T lane-instructions / s
        timed = {n: v for n, v in kernels.items() if n in ALG and v["launches"]}

        def kernel_roofline(name, v):
            per_ms = v["ms"] / v["launches"]
            if name in issue:  # 0.25 B/base in, every start position tested: instruction issue is the bound
                positions = n_rows_total if name == "collect_owned" else rows_tested_r  # every GPU tests every position
                ach = issue[name] * positions / per_ms / 1e9
                return {"bound": "issue", "ms_per_launch": per_ms, "achieved": ach, "peak": issue_peak,
                        "unit": "T lane-instr/s", "frac": ach / issue_peak,
                        "instructions_per_position": issue[name], "positions_per_launch": positions,
                        "hbm_gbs": ALG[name] / per_ms / 1e6, "hbm_frac": ALG[name] / per_ms / 1e6 / peak}
            return {"bound": "hbm", "ms_per_launch": per_ms, "achieved": ALG[name] / per_ms / 1e6, "peak": peak,
                    "unit": "GB/s", "frac": ALG[name] / per_ms / 1e6 / peak}
        roofline = None
        if timed:
            dom = max(timed, key=lambda n: timed[n]["ms"])
            d = timed[dom]
            r = kernel_roofline(dom, d)
            traffic = None
            try:
                with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                    traffic = json.load(f).get(f"{args.workload}:n{world}:{dom}")
            except Exception:
                pass
            pipe_bytes = sum(ALG[n] * v["launches"] / args.steps for n, v in timed.items())
            roofline = {"bound": r["bound"], "kernel": dom, "achieved": r["achieved"], "peak": r["peak"],
                        "unit": r["unit"], "frac": r["frac"], "traffic": traffic, "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": ALG[dom], "ms_per_launch": r["ms_per_launch"],
                        "share_of_step": d["ms"] / ms,
                        "pipeline": {"algorithmic_bytes_per_step": pipe_bytes,
                                     "bytes_per_kmer": pipe_bytes / max(rows_r, 1),
                                     "achieved": pipe_bytes / (ms / args.steps) / 1e6,
                                     "frac": pipe_bytes / (ms / args.steps) / 1e6 / peak,
                                     "note": "all kernels of one step on this rank / whole step time"},
                        "per_kernel": {n: kernel_roofline(n, v) for n, v in timed.items()}}
            if r["bound"] == "issue":
                roofline.update({q: r[q] for q in ("instructions_per_position", "positions_per_launch", "hbm_gbs",
                                                   "hbm_frac")})
            if gather:  # bases read from the other GPUs' shards, per step and rank, against the NVLink peer rate
                nv = 8.0 * (n_words_total - n_words_local)
                own = timed.get("collect_owned")
                if own:
                    per = own["ms"] / own["launches"]
                    roofline["nvlink"] = {"bytes_per_launch": nv, "achieved": nv / per / 1e6, "peak": NVLINK_PEER_GBS,
                                          "unit": "GB/s", "frac": nv / per / 1e6 / NVLINK_PEER_GBS,
                                          "note": "2-bit packed bases read through peer memory inside collect_owned; "
                                                  "routing 8-byte k-mers instead would move 8*(G-1)/G B per k-mer"}
        cpu, one = cpu_baselines(n_bases, k, seed, reads, args.cpu_sample, 1_000_000)
        par = {"gather": "base-range shards (one per GPU, (k-1)-base overlap) mapped into every GPU; each GPU reads all "
                         "shards over NVLink and counts the k-mers it owns (dnagpu_owner_of); no k-mer exchange, one "
                         "3-element all-reduce",
               "peer": "base-range shards, k-mers routed to owner GPUs by hash: level-1 scatter kernel stores into the "
                       "owners' memory over NVLink, no all-to-all",
               "fused": "base-range shards, k-mers routed to owner GPUs by hash: level-1 layout + one NCCL all-to-all",
               "routed": "base-range shards, dnagpu_partition + NCCL all-to-all + dnagpu_count_keys"}
        e2e_api = ("dnagpu_count_reads(ctx, host_words, n_reads, 150, 5, k, &where, &stats, NULL)" if reads and world == 1 else
                   "dnagpu_count_kmers(ctx, host_words, n_bases, k, NULL, &stats, NULL)" if world == 1 else
                   "per rank and step: pinned host shard -> H2D into its peer-mapped ring buffer, barrier, "
                   "dnagpu.distributed.count_sharded_gather (dnagpu_count with an owner restriction), all-reduce"
                   + ("; two rings: the H2D of step s + 1 overlaps the count of step s" if e2e_overlapped else "")
                   if gather else
                   "per rank: dnagpu_seq_upload* of its shard + dnagpu.distributed.count_sharded_" + args.exchange)
        line = {
            "metric": METRIC, "value": value, "unit": "Gkmer/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": desc, "n_bases": n_bases, "k": k, "seed": seed,
                       "unit_of_value": "k-mers generated and tested per second" if reads else "k-mers counted per second",
                       "repeat_every": REPEAT_EVERY, "block_bases": 1024,
                       "l2": "inputs (packed words + partition buffers) larger than L2; no flush needed"
                       if n_bases >= 100_000_000 else "input smaller than L2 (the reference's own CPU-sized case)",
                       "parallelism": "single GPU" if world == 1 else f"{world} GPUs, exchange={args.exchange}: " + par[args.exchange],
                       "load_factor": args.load_factor or 0.5},
            "result": {"total": stats[0], "distinct": stats[1], "unique": stats[2],
                       "oracle": "equal to tests/golden/big_expected.json (CPU oracle at the full size)"
                       if gold is not None else "not compared (size overridden or no golden entry)"},
            "e2e": {"value": e2e_value, "unit": "Gkmer/s", "steps": args.e2e_steps,
                    "ms_per_step": 1e3 * e2e_s / args.e2e_steps,
                    "h2d_bytes_per_step": int(8 * n_words_total), "d2h_bytes_per_step": 24 * world, "api": e2e_api},
            "gpu_launches": launches, "kernels": kernels, "roofline": roofline, "cpu_baseline": cpu,
            "cpu_baseline_1thread": one, "extract": extract, "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if px is not None:
        px.close()
    if ring is not None:
        ring.close()
    seq.free()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of the resident-input leg (every k of c5) and launches of the extraction leg; "
                         "the host-buffer leg runs --e2e-steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--k", type=int, default=0, help="override k (c5: one k of the sweep instead of all 30)")
    ap.add_argument("--n-bases", type=int, default=0, help="override the workload size (debugging)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--load-factor", type=float, default=0.0)
    ap.add_argument("--cpu-sample", type=int, default=16_000_000)
    ap.add_argument("--cpu-large-sample", type=int, default=0,
                    help="--impl reference: bases per step (e.g. 100000000: a table that no longer fits the CPU caches)")
    ap.add_argument("--no-extract", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the timed legs returned in their last step as DIR/<name>.npy (float64)")
    ap.add_argument("--planes", action="store_true",
                    help="reads workload, N = 1: evaluate the WHERE clause with the plane test (DNAGPU_WHERE_FLAG_PLANES)")
    ap.add_argument("--chunks", type=int, default=4, help="--exchange fused: digit sub-ranges the exchange is pipelined in")
    ap.add_argument("--exchange", default="gather", choices=["gather", "peer", "fused", "routed"],
                    help="N > 1: gather = every GPU reads all shards over NVLink and counts the k-mers it owns; "
                         "peer = scatter kernel stores routed k-mers into the owners' memory; fused = level-1 layout + "
                         "NCCL all-to-all; routed = separate dnagpu_partition pass")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
