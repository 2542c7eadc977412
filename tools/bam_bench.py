#!/usr/bin/env python3
"""Cost of unaligned BAM output (ssc_set_option "bam") beside BGZF FASTQ, on bench.py's job and on a generic-kernel profile.

Profiles:
  XTen       bench.write_job's 3 Gb x 30x job (the fast kernel, RL 151)
  rl250_b31  bench.write_job's genome at --generic-genome-bases with a synthetic K = 3 PE profile at RL 250 (the generic kernel)
One handle per profile, --batch-pairs pairs per batch.  Both outputs are one stream of both mates: "bgzf" is gzip + bgzf +
interleave (BGZF FASTQ), "bam" the BGZF blocks of BAM records.  Arms, each alternated between the two outputs on the same handle
(the order flips every round; every round takes the next span of --batches batches, the same span for both outputs of an arm):
  device  ssc_generate_device, the compressed slabs left on the device
  file    ssc_generate end to end into one file through libsimuscop_host's ssh_writer (4 threads, the CLI's default) with
          ssh_writer_bgzf; for BAM the ssc_bam_header block first, as the CLI writes it
A call is timed with the host clock from a synchronised device to its return (file: to ssh_writer_close); the call of one
ticket before it, untimed, takes the re-sizing of the slabs and the refit of the Huffman table that a switch of the format
causes.  Prints one JSON line per profile: Gbases/s per round, the median of every (arm, output), the CUDA-event time per call of
the generation kernel and of the compression (deflate + pass 2, ssc_stats compact_kernel_ms) on the device arm, compressed
bytes per base and raw bytes per read of each output, and the card's name and power limit read in the same run.  The files go to
--workdir and are deleted after each call (page cache: the writes are not synced).

  python tools/bam_bench.py [--profile XTen] [--batches 8] [--rounds 5]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bgzf_bench import writer_lib  # noqa: E402
from interleave_bench import card  # noqa: E402

OUTPUTS = ("bgzf", "bam")


def config(a, profile):
    import bench
    from simuscop_b200 import synth
    if profile == "XTen":
        return bench.write_job(a.workdir, a.genome_bases, a.coverage, profile)[0]
    bench.write_job(a.workdir, a.generic_genome_bases, a.coverage)             # the FASTA (cached per box)
    prof = os.path.join(a.workdir, "bam_rl250.profile")
    synth.write_profile(prof, seed=250, kmer=3, read_length=250, bins=31, n_live_qual=12)
    cfg = os.path.join(a.workdir, "bam_rl250_%d_%d.txt" % (a.generic_genome_bases, a.coverage))
    synth.write_config(cfg, ref=os.path.join(a.workdir, "genome_%d.fa" % a.generic_genome_bases), profile=prof, name="test",
                       output=os.path.join(a.workdir, "out"), layout="PE", threads=1, verbose=0, coverage=a.coverage,
                       insertSize=400)
    return cfg


def run_profile(a, profile):
    import torch
    from simuscop_b200 import cuda_binding, host_binding
    job = host_binding.Job(config(a, profile), 1)
    gen = cuda_binding.Generator(0)
    hl, sink = writer_lib()
    out = os.path.join(a.workdir, "bam_bench_out")
    os.makedirs(out, exist_ok=True)
    header = cuda_binding.bam_header("test")
    try:
        gen.set_option("batch_pairs", a.batch_pairs)
        gen.set_option("interleave", 1)
        gen.set_option("bgzf", 1)
        gen.set_read_group("test")
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

        def to_file(bam, lo, hi):
            path = os.path.join(out, "r.bam" if bam else "r.fq.gz")
            w = C.c_void_p()
            if hl.ssh_writer_open(path.encode(), None, 4, C.byref(w)) or hl.ssh_writer_bgzf(w, None, None):
                raise RuntimeError("can not open %s" % path)
            if bam and sink(w, header, len(header), None, 0, 0, 0):
                raise RuntimeError("writing the header failed")
            gen.generate(lo, hi, sink=sink, user=w)
            if hl.ssh_writer_close(w, None, None):
                raise RuntimeError("writing %s failed" % path)
            os.unlink(path)

        def timed(arm, output, lo, hi):
            gen.set_option("bam", int(output == "bam"))
            gen.set_option("gzip", int(output == "bgzf"))
            gen.generate_device(lo, lo + 32)
            torch.cuda.synchronize()
            gen.reset_stats()
            t0 = time.perf_counter()
            if arm == "file":
                to_file(output == "bam", lo, hi)
            else:
                gen.generate_device(lo, hi)
            dt = time.perf_counter() - t0
            return gen.stats(), dt

        arms = ("device", "file")
        lo, hi = span(1)
        for arm in arms:                                    # warm-up: the slabs of both outputs allocated
            for output in OUTPUTS:
                timed(arm, output, lo, hi)
        rates = {arm: {o: [] for o in OUTPUTS} for arm in arms}
        per_base = {o: [] for o in OUTPUTS}
        raw_per_read = {o: [] for o in OUTPUTS}
        kernel_ms = {o: {"gen": [], "compress": []} for o in OUTPUTS}
        kernel = None
        for r in range(a.rounds):
            for arm in arms:
                lo, hi = span(a.batches)
                for output in (OUTPUTS if r % 2 == 0 else OUTPUTS[::-1]):
                    st, dt = timed(arm, output, lo, hi)
                    rates[arm][output].append(round(st["bases_emitted"] / dt / 1e9, 2))
                    if arm == "device":
                        per_base[output].append(round(st["gz_bytes"] / st["bases_emitted"], 5))
                        raw_per_read[output].append(round(st["fastq_bytes"] / st["reads_emitted"], 2))
                        kernel_ms[output]["gen"].append(round(st["gen_kernel_ms"], 2))
                        kernel_ms[output]["compress"].append(round(st["compact_kernel_ms"], 2))
                        kernel = (st["gen_kernel"], st["gen_nch"], st["gen_qmode"])
        med = {arm: {k: statistics.median(v) for k, v in d.items()} for arm, d in rates.items()}
        return {"profile": profile, "read_length": job.read_length,
                "genome_bases": a.genome_bases if profile == "XTen" else a.generic_genome_bases, "coverage": a.coverage,
                "batch_pairs": bp, "batches_per_call": a.batches, "gen_kernel_nch_qmode": kernel, "gbases_per_s": rates,
                "median_gbases_per_s": med, "bam_over_bgzf_device": round(med["device"]["bam"] / med["device"]["bgzf"], 4),
                "compressed_bytes_per_base": {k: statistics.median(v) for k, v in per_base.items()},
                "raw_bytes_per_read": {k: statistics.median(v) for k, v in raw_per_read.items()},
                "median_kernel_ms_per_call": {o: {k: statistics.median(v) for k, v in d.items()} for o, d in kernel_ms.items()},
                "card": card()}
    finally:
        gen.close()
        job.close()
        if os.path.isdir(out):
            for f in os.listdir(out):
                os.unlink(os.path.join(out, f))
            os.rmdir(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--profile", action="append", choices=["XTen", "rl250_b31"])
    ap.add_argument("--batches", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch-pairs", type=int, default=1 << 20)
    ap.add_argument("--genome-bases", type=int, default=3000000000)
    ap.add_argument("--generic-genome-bases", type=int, default=300000000)
    ap.add_argument("--coverage", type=int, default=30)
    ap.add_argument("--workdir", default=os.environ.get("SIMUSCOP_BENCH_DIR", "/tmp/simuscop_bench"))
    a = ap.parse_args()
    import torch
    import __graft_entry__ as ge
    ge.build()
    os.makedirs(a.workdir, exist_ok=True)
    torch.cuda.init()
    for profile in a.profile or ["XTen", "rl250_b31"]:
        print(json.dumps(run_profile(a, profile)), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
