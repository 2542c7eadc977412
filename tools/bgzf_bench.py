#!/usr/bin/env python3
"""Cost of BGZF output (ssc_set_option "bgzf") beside plain multi-member gzip, on bench.py's job.

One handle, bench.write_job's 3 Gb x 30x job for the profile, --batch-pairs pairs per batch.  Arms, each alternated between
gzip and gzip + bgzf on the same handle (the order flips every round; every round takes the next span of --batches batches of
the job, the same span for both outputs of an arm):
  device  ssc_generate_device, the compressed slabs left on the device
  files   ssc_generate end to end into two files through libsimuscop_host's ssh_writer (4 threads, the CLI's default); with
          bgzf the writer walks the blocks, writes both .gzi indexes and appends the EOF blocks (ssh_writer_bgzf)
A call is timed with the host clock from a synchronised device to its return (files: to ssh_writer_close); the call of one
ticket before it, untimed, takes the re-sizing of the slabs that a switch of the mode causes.  The size ratio is gz_bytes of
bgzf over gzip for the same span.  Prints one JSON line per profile: Gbases/s per round, the median of every (arm, mode), the
size ratios and the card's name and power limit read in the same run.  The files go to --workdir and are deleted after each
call (page cache: the writes are not synced).

  python tools/bgzf_bench.py [--profile XTen] [--batches 8] [--rounds 5]
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

from interleave_bench import card  # noqa: E402


def writer_lib():
    from simuscop_b200 import abi, host_binding
    hl = host_binding.lib()
    hl.ssh_writer_open.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]
    hl.ssh_writer_bgzf.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
    hl.ssh_writer_sink.restype = C.c_void_p
    hl.ssh_writer_close.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    return hl, C.cast(hl.ssh_writer_sink(), abi.SINK_FN)


def run_profile(a, profile):
    import torch
    import bench
    from simuscop_b200 import cuda_binding, host_binding
    cfg, _ = bench.write_job(a.workdir, a.genome_bases, a.coverage, profile)
    job = host_binding.Job(cfg, 1)
    gen = cuda_binding.Generator(0)
    hl, sink = writer_lib()
    out = os.path.join(a.workdir, "bgzf_bench_out")
    os.makedirs(out, exist_ok=True)
    try:
        gen.set_option("batch_pairs", a.batch_pairs)
        gen.set_option("gzip", 1)
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

        def to_files(bgzf, lo, hi):
            paths = [os.path.join(out, "r_%d.fq.gz" % k) for k in (1, 2)]
            w = C.c_void_p()
            if hl.ssh_writer_open(paths[0].encode(), paths[1].encode(), 4, C.byref(w)):
                raise RuntimeError("can not open %s" % paths[0])
            if bgzf and hl.ssh_writer_bgzf(w, (paths[0] + ".gzi").encode(), (paths[1] + ".gzi").encode()):
                raise RuntimeError("ssh_writer_bgzf failed")
            gen.generate(lo, hi, sink=sink, user=w)
            if hl.ssh_writer_close(w, None, None):
                raise RuntimeError("writing %s failed" % paths[0])

        def cleanup():
            for f in os.listdir(out):
                os.unlink(os.path.join(out, f))

        def timed(arm, bgzf, lo, hi):
            gen.set_option("bgzf", int(bgzf))
            # a switch of the mode re-sizes the slabs (a stored block is 8 bytes longer) at the next call: a call of one ticket
            # does that outside the timed region
            if arm == "files":
                gen.generate(lo, lo + 32, sink=lambda *x: 0)
            else:
                gen.generate_device(lo, lo + 32)
            torch.cuda.synchronize()
            gen.reset_stats()
            t0 = time.perf_counter()
            if arm == "files":
                to_files(bgzf, lo, hi)
            else:
                gen.generate_device(lo, hi)
            dt = time.perf_counter() - t0
            st = gen.stats()
            if arm == "files":
                cleanup()
            return st["bases_emitted"] / dt / 1e9, st["gz_bytes"]

        arms = ("device", "files")
        lo, hi = span(1)
        for arm in arms:                                    # warm-up: slabs of both modes allocated, gzip table fitted
            for bgzf in (False, True):
                timed(arm, bgzf, lo, hi)
        rates = {arm: {"gzip": [], "bgzf": []} for arm in arms}
        ratios = []
        for r in range(a.rounds):
            for arm in arms:
                lo, hi = span(a.batches)
                order = (False, True) if r % 2 == 0 else (True, False)
                size = {}
                for bgzf in order:
                    g, size[bgzf] = timed(arm, bgzf, lo, hi)
                    rates[arm]["bgzf" if bgzf else "gzip"].append(round(g, 2))
                ratios.append(round(size[True] / size[False], 5))
        med = {arm: {k: statistics.median(v) for k, v in d.items()} for arm, d in rates.items()}
        return {"profile": profile, "read_length": job.read_length, "batch_pairs": bp, "batches_per_call": a.batches,
                "gbases_per_s": rates, "median_gbases_per_s": med, "bgzf_over_gzip_bytes": ratios, "card": card()}
    finally:
        gen.close()
        job.close()
        if os.path.isdir(out):
            for f in os.listdir(out):
                os.unlink(os.path.join(out, f))
            os.rmdir(out)


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
