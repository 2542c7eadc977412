#!/usr/bin/env python3
"""Plain, gzip and gzip + BGZF output of the generic generation kernel, device-resident.

bench.write_job's genome (--genome-bases, --coverage) with two synthetic K = 3 PE profiles the fast kernel does not take:
  rl250_b31  RL 250, 31 bins: the substitution tables in shared memory (generate_kernel<K3 = true>)
  rl320_b76  RL 320, 76 bins: the tables in global memory (generate_kernel<K3 = false>)
One handle per profile, --batch-pairs pairs per batch.  Every round takes the next span of --batches batches and runs
ssc_generate_device on it in each mode, the order rotating by round; a call is timed with the host clock from a synchronised
device to its return.  A call of one ticket before each timed call, untimed, takes the re-sizing of the slabs and the blob
scratch that a switch of the mode causes.  The compression ratio is gz_bytes over fastq_bytes of the same span.  Prints one
JSON line per profile: Gbases/s per round and mode, their medians, the ratios, the instance that ran, and the card's name and
power limit read in the same run.

  python tools/generic_gzip_bench.py [--batches 4] [--rounds 5] [--genome-bases 300000000]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from interleave_bench import card  # noqa: E402

PROFILES = {"rl250_b31": dict(read_length=250, bins=31, n_live_qual=12, insert=400),
            "rl320_b76": dict(read_length=320, bins=76, n_live_qual=7, insert=500)}
MODES = ("plain", "gzip", "bgzf")


def write_config(a, name):
    import bench
    from simuscop_b200 import synth
    spec = PROFILES[name]
    bench.write_job(a.workdir, a.genome_bases, a.coverage)            # the FASTA (cached per box)
    prof = os.path.join(a.workdir, "generic_gzip_%s.profile" % name)
    synth.write_profile(prof, seed=spec["read_length"], kmer=3, read_length=spec["read_length"], bins=spec["bins"],
                        n_live_qual=spec["n_live_qual"])
    cfg = os.path.join(a.workdir, "generic_gzip_%s_%d_%d.txt" % (name, a.genome_bases, a.coverage))
    synth.write_config(cfg, ref=os.path.join(a.workdir, "genome_%d.fa" % a.genome_bases), profile=prof, name="test",
                       output=os.path.join(a.workdir, "out"), layout="PE", threads=1, verbose=0, coverage=a.coverage,
                       insertSize=spec["insert"])
    return cfg


def run_profile(a, name):
    import torch
    from simuscop_b200 import cuda_binding, host_binding
    job = host_binding.Job(write_config(a, name), 1)
    gen = cuda_binding.Generator(0)
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

        def timed(mode, lo, hi):
            gen.set_option("gzip", int(mode != "plain"))
            gen.set_option("bgzf", int(mode == "bgzf"))
            gen.generate_device(lo, lo + 32)
            torch.cuda.synchronize()
            gen.reset_stats()
            t0 = time.perf_counter()
            gen.generate_device(lo, hi)
            dt = time.perf_counter() - t0
            st = gen.stats()
            return st["bases_emitted"] / dt / 1e9, st

        lo, hi = span(1)
        for mode in MODES:                                  # warm-up: every mode's buffers, the gzip table fitted
            timed(mode, lo, hi)
        rates = {m: [] for m in MODES}
        ratios = {"gzip": [], "bgzf": []}
        kernel = None
        for r in range(a.rounds):
            lo, hi = span(a.batches)
            order = MODES[r % 3:] + MODES[:r % 3]
            for mode in order:
                g, st = timed(mode, lo, hi)
                rates[mode].append(round(g, 2))
                if mode != "plain":
                    ratios[mode].append(round(st["gz_bytes"] / st["fastq_bytes"], 5))
                kernel = (st["gen_kernel"], st["gen_nch"], st["gen_smem_bytes"])
        med = {k: statistics.median(v) for k, v in rates.items()}
        return {"profile": name, "read_length": PROFILES[name]["read_length"], "bins": PROFILES[name]["bins"],
                "genome_bases": a.genome_bases, "coverage": a.coverage, "batch_pairs": bp, "batches_per_call": a.batches,
                "gen_kernel_nch_smem": kernel, "gbases_per_s": rates, "median_gbases_per_s": med,
                "compressed_over_fastq_bytes": ratios,
                "median_compressed_over_fastq_bytes": {k: statistics.median(v) for k, v in ratios.items()}, "card": card()}
    finally:
        gen.close()
        job.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--profile", action="append", choices=sorted(PROFILES))
    ap.add_argument("--batches", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch-pairs", type=int, default=1 << 20)
    ap.add_argument("--genome-bases", type=int, default=300000000)
    ap.add_argument("--coverage", type=int, default=30)
    ap.add_argument("--workdir", default=os.environ.get("SIMUSCOP_BENCH_DIR", "/tmp/simuscop_bench"))
    a = ap.parse_args()
    import torch
    import __graft_entry__ as ge
    ge.build()
    os.makedirs(a.workdir, exist_ok=True)
    torch.cuda.init()
    for name in a.profile or sorted(PROFILES):
        print(json.dumps(run_profile(a, name)), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
