#!/usr/bin/env python3
"""Rate of interleaved paired-end output (ssc_set_option "interleave") beside two-file output, on bench.py's job.

One handle, bench.write_job's 3 Gb x 30x job for the profile, --batch-pairs pairs per batch.  Arms, each alternated between
two-file and interleaved output on the same handle (the order flips every round; every round takes the next span of
--batches batches of the job, the same span for both outputs of an arm):
  device       ssc_generate_device, plain FASTQ left in the device slabs
  device_gzip  the same with the gzip option
  host         ssc_generate end to end into a host sink that discards the slabs (kernels, pass 2, device->host copies)
A call is timed with the host clock from a synchronised device to its return; the call of one ticket before it, untimed, takes
the re-sizing of the slabs that a switch of the output mode causes.  Prints one JSON line per profile: Gbases/s per
round and the median of every (arm, output), the card's name and power limit read in the same run.  Disk writes are not
measured here.

  python tools/interleave_bench.py [--profile XTen --profile GAIIx] [--batches 8] [--rounds 5]
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
    from simuscop_b200 import abi, cuda_binding, host_binding
    cfg, _ = bench.write_job(a.workdir, a.genome_bases, a.coverage, profile)
    job = host_binding.Job(cfg, 1)
    gen = cuda_binding.Generator(0)
    discard = abi.SINK_FN(lambda user, b1, l1, b2, l2, first, n: 0)
    try:
        gen.set_option("batch_pairs", a.batch_pairs)
        planned, _ = job.prepare(0, gen)
        bp = a.batch_pairs
        nbatch = planned // bp
        if a.batches + 1 > nbatch:
            raise SystemExit("the job has %d batches of %d pairs" % (nbatch, bp))
        first = 0

        def span(n):
            nonlocal first
            if first + n > nbatch:
                first = 0
            first += n
            return (first - n) * bp, first * bp

        def timed(arm, interleave, lo, hi):
            gen.set_option("interleave", int(interleave))
            gen.set_option("gzip", int(arm == "device_gzip"))
            # a switch of the output mode re-sizes the slabs (device and pinned host memory) at the next call: a call of one
            # ticket does that outside the timed region
            if arm == "host":
                gen.generate(lo, lo + 32, sink=discard)
            else:
                gen.generate_device(lo, lo + 32)
            torch.cuda.synchronize()
            gen.reset_stats()
            t0 = time.perf_counter()
            if arm == "host":
                gen.generate(lo, hi, sink=discard)
            else:
                gen.generate_device(lo, hi)
            dt = time.perf_counter() - t0
            return gen.stats()["bases_emitted"] / dt / 1e9

        arms = ("device", "device_gzip", "host")
        lo, hi = span(1)
        for arm in arms:                                    # warm-up: slabs of every mode allocated, gzip table fitted
            for ilv in (False, True):
                timed(arm, ilv, lo, hi)
        rates = {arm: {"two_files": [], "interleaved": []} for arm in arms}
        for r in range(a.rounds):
            for arm in arms:
                lo, hi = span(a.batches)
                order = (False, True) if r % 2 == 0 else (True, False)
                for ilv in order:
                    rates[arm]["interleaved" if ilv else "two_files"].append(round(timed(arm, ilv, lo, hi), 2))
        med = {arm: {k: statistics.median(v) for k, v in d.items()} for arm, d in rates.items()}
        return {"profile": profile, "read_length": job.read_length, "batch_pairs": bp, "batches_per_call": a.batches,
                "gbases_per_s": rates, "median_gbases_per_s": med, "card": card()}
    finally:
        gen.close()
        job.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--profile", action="append", choices=["GAIIx", "HiSeq2000", "HiSeq2500", "XTen"])
    ap.add_argument("--batches", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch-pairs", type=int, default=1 << 20)
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
