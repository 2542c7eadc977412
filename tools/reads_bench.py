#!/usr/bin/env python3
"""Rate of the array output (ssc_generate_reads) beside the device-resident FASTQ mode (ssc_generate_device) on bench.py's job.

One handle, bench.write_job's 3 Gb x 30x job for the profile, --batch-pairs pairs per batch.  After a warm-up of both calls,
--rounds rounds each time the same span of --batches batches through both calls, alternating which goes first; every round
takes the next span of the job, so no call reads what a recent one wrote.  A call is timed with the host clock from a
synchronised device to its return (both calls return when their output is complete).  Prints one JSON line per profile:
Gbases/s per round and the median of each arm, the card and its power limit.

  python tools/reads_bench.py [--profile XTen --profile GAIIx ...] [--batches 8] [--rounds 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except Exception as ex:
        return "unknown (%s)" % type(ex).__name__


def run_profile(a, profile):
    import torch
    import bench
    from simuscop_b200 import cuda_binding, host_binding
    cfg, _ = bench.write_job(a.workdir, a.genome_bases, a.coverage, profile)
    job = host_binding.Job(cfg, 1)
    gen = cuda_binding.Generator(0)
    try:
        gen.set_option("batch_pairs", a.batch_pairs)
        planned, _ = job.prepare(0, gen)
        bp = a.batch_pairs
        nbatch = planned // bp
        if a.batches + 1 > nbatch:
            raise SystemExit("the job has %d batches of %d pairs" % (nbatch, bp))
        out = gen.empty_reads(a.batches * bp)
        first = 0

        def span(n):
            nonlocal first
            if first + n > nbatch:
                first = 0
            first += n
            return (first - n) * bp, first * bp

        def timed(kind, lo, hi):
            torch.cuda.synchronize()
            gen.reset_stats()
            t0 = time.perf_counter()
            if kind == "reads":
                gen.generate_reads(lo, hi, out=out)
            else:
                gen.generate_device(lo, hi)
            dt = time.perf_counter() - t0
            return gen.stats()["bases_emitted"] / dt / 1e9

        lo, hi = span(1)
        timed("reads", lo, hi)
        timed("device", lo, hi)
        rates = {"reads": [], "device": []}
        for r in range(a.rounds):
            lo, hi = span(a.batches)
            for kind in (("reads", "device") if r % 2 == 0 else ("device", "reads")):
                rates[kind].append(round(timed(kind, lo, hi), 2))
        return {"profile": profile, "batch_pairs": bp, "batches_per_call": a.batches, "gbases_per_s": rates,
                "median_gbases_per_s": {k: statistics.median(v) for k, v in rates.items()},
                "card": card()}
    finally:
        gen.close()
        job.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--profile", action="append", choices=["GAIIx", "HiSeq2000", "HiSeq2500", "XTen"])
    ap.add_argument("--batches", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch-pairs", type=int, default=1 << 21)
    ap.add_argument("--genome-bases", type=int, default=3000000000)
    ap.add_argument("--coverage", type=int, default=30)
    ap.add_argument("--workdir", default=os.environ.get("SIMUSCOP_BENCH_DIR", "/tmp/simuscop_bench"))
    a = ap.parse_args()
    import torch
    import __graft_entry__ as ge
    ge.build()
    os.makedirs(a.workdir, exist_ok=True)
    torch.cuda.init()
    for profile in a.profile or ["XTen"]:
        print(json.dumps(run_profile(a, profile)), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
