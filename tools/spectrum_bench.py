"""Cost of the k-mer abundance spectrum against the plain count and against today's table route.

For each workload, on one device-resident synthetic sequence (include/dnagpu_synth.h, the seeds of bench.py):
  count     dnagpu_count, aggregates only (the headline query)
  spectrum  dnagpu_count_spectrum with H = --max-count (the same count with the spectrum binned on the way)
  table     dnagpu_count with the (kmer, count) table, then torch.bincount(clamp(counts, max=H)) on the device:
            the way to get the spectrum without this feature
The three are timed in turn, --reps times each after --warmup rounds, with CUDA events on the stream the library
shares with torch (every call ends in a stream synchronise).  The spectrum is checked against the table route once.
One JSON line per workload on stdout (and appended to --out), with the card's name and power limit."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "dna-sequences-pg-extension_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dnagpu  # noqa: E402

WORKLOADS = {  # name: (n_bases, k, seed)
    "c4": (3_100_000_000, 31, 4),      # BASELINE configs[3]: partition path, the headline workload
    "c2": (100_000_000, 21, 2),        # BASELINE configs[1]
    "dense_k10": (1_000_000_000, 10, 5),  # 1 Gbp at k = 10: dense counters
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, check=True).stdout.strip()
        name, power, clock = (s.strip() for s in out.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except (OSError, subprocess.CalledProcessError, ValueError):
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown", "max_sm_clock": "unknown"}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--max-count", type=int, default=10_000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("spectrum_bench: no CUDA device")
    H = args.max_count
    info = card()
    ctx = dnagpu.Context(0, torch_stream=True)
    for name in args.workloads.split(","):
        n, k, seed = WORKLOADS[name]
        seq = ctx.synth(n, seed, 8)

        def count():
            return ctx.count(seq, k)[0]

        def spectrum():
            return ctx.count_spectrum(seq, k, max_count=H)

        def table_route():
            st, table = ctx.count(seq, k, table=True)
            _, addr = table.device_pointers()
            counts = dnagpu._device_view(addr, table.rows, 0)
            hist = torch.bincount(torch.clamp(counts, max=H), minlength=H + 1)[1:]
            return st, table, hist

        legs = {"count": count, "spectrum": spectrum, "table": table_route}
        times = {leg: [] for leg in legs}
        check = None
        for r in range(args.warmup + args.reps):
            for leg, fn in legs.items():
                ms, out = timed(fn)
                if leg == "table":
                    st, table, hist = out
                    if check is None:
                        check = hist.cpu().numpy().astype(np.uint64)
                    table.free()
                    del hist
                elif leg == "spectrum":
                    st, spec = out
                if r >= args.warmup:
                    times[leg].append(ms)
        same = bool(np.array_equal(spec, check)) and int(spec.sum()) == st.distinct
        seq.free()
        med = {leg: statistics.median(v) for leg, v in times.items()}
        rec = {"workload": name, "n_bases": n, "k": k, "max_count": H, **info,
               "count_ms": round(med["count"], 3), "spectrum_ms": round(med["spectrum"], 3),
               "table_bincount_ms": round(med["table"], 3),
               "spectrum_over_count": round(med["spectrum"] / med["count"], 4),
               "table_over_spectrum": round(med["table"] / med["spectrum"], 3),
               "count_ms_all": [round(x, 3) for x in times["count"]],
               "spectrum_ms_all": [round(x, 3) for x in times["spectrum"]],
               "table_bincount_ms_all": [round(x, 3) for x in times["table"]],
               "distinct": int(st.distinct), "spectrum_equals_table_route": same,
               "timing": f"CUDA events, median of {args.reps} after {args.warmup} warm-up rounds, legs alternated"}
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
        if not same:
            sys.exit(f"{name}: the spectrum differs from the table route")
    ctx.close()


if __name__ == "__main__":
    main()
