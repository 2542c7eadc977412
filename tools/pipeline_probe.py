#!/usr/bin/env python3
"""Where the time of a step of the device-resident pipeline goes, batch by batch, on bench.py's job.

One ssc_generate_device call over --batches batches runs under torch.profiler, whose CUDA activity trace (CUPTI) times every
kernel and memset on the stream it ran on.  Per batch k it prints:
  setup  the memsets and locate_kernel before generation launch k, from the first of them to the launch's start
  wait   the compute stream's idle time between generation launch k-1's end and that set-up (the mover it waits for, and on
         builds that scan on the compute stream, the scan)
  gen    generate_slots_kernel of batch k
  scan   scan_blobs_kernel of batch k, and the stream it ran on
  move   the concurrent mover's move_blobs_tma_kernel of batch k (it runs under generation launch k+1)
  step   start of generation launch k+1 - start of launch k
  slack  end of generation launch k+1 - end of the move of batch k: > 0 when the mover leg finished under that launch
A summary line follows (medians over the batches with a predecessor and a successor), beside the same call's ssc_stats
averages (CUDA events inside the library) and the step time of an unprofiled call, the card and its power limit.

  python tools/pipeline_probe.py [--batches 24] [--opts concurrent_move=9 --opts concurrent_move=10 ...]

Each --opts is one run (comma-separated ssc_set_option settings) on the same handle; without it, one run with the defaults.
"""
import argparse
import glob
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def kernel_events(trace):
    """(kind, stream, start_us, end_us) of the pipeline's kernels and memsets in a chrome trace, in start order."""
    kinds = (("generate_slots_kernel", "gen"), ("scan_blobs_kernel", "scan"), ("move_blobs_tma_kernel", "move"),
             ("move_blobs_kernel", "standalone_move"), ("locate_kernel", "setup"))
    out = []
    for e in trace.get("traceEvents", []):
        if e.get("ph") != "X" or e.get("cat") not in ("kernel", "gpu_memset"):
            continue
        kind = "setup" if e["cat"] == "gpu_memset" else next((k for n, k in kinds if n in e.get("name", "")), None)
        if kind:
            out.append((kind, e.get("args", {}).get("stream"), float(e["ts"]), float(e["ts"]) + float(e["dur"])))
    return sorted(out, key=lambda x: x[2])


def per_batch(events):
    """One dict per generation launch (see the module text); times in ms."""
    gens = [e for e in events if e[0] == "gen"]
    if not gens:
        raise SystemExit("no generate_slots_kernel in the CUDA activity trace: the profiler did not see the library's kernels")
    scans = [e for e in events if e[0] == "scan"]
    moves = [e for e in events if e[0] == "move"]
    rows = []
    for k, g in enumerate(gens):
        lo = gens[k - 1][3] if k else float("-inf")
        setup = [e for e in events if e[0] == "setup" and e[1] == g[1] and lo <= e[2] < g[2]]
        r = {"batch": k, "gen": (g[3] - g[2]) / 1e3}
        if setup:
            r["setup"] = (g[2] - setup[0][2]) / 1e3
            if k:
                r["wait"] = (setup[0][2] - lo) / 1e3
        if k < len(scans):
            r["scan"] = (scans[k][3] - scans[k][2]) / 1e3
            r["scan_stream"] = "compute" if scans[k][1] == g[1] else "other"
        if k < len(moves):
            r["move"] = (moves[k][3] - moves[k][2]) / 1e3
            if k + 1 < len(gens):
                r["slack"] = (gens[k + 1][3] - moves[k][3]) / 1e3
        if k + 1 < len(gens):
            r["step"] = (gens[k + 1][2] - g[2]) / 1e3
        rows.append(r)
    return rows


def summary(rows):
    inner = rows[1:-1] or rows
    out = {}
    for key in ("setup", "wait", "gen", "scan", "move", "step", "slack"):
        v = [r[key] for r in inner if key in r]
        if v:
            out[key] = round(statistics.median(v), 4)
    out["scan_stream"] = sorted({r["scan_stream"] for r in inner if "scan_stream" in r})
    return out


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except Exception as ex:
        return "unknown (%s)" % type(ex).__name__


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch-pairs", type=int, default=1 << 21)
    ap.add_argument("--genome-bases", type=int, default=3000000000)
    ap.add_argument("--coverage", type=int, default=30)
    ap.add_argument("--profile", default="XTen", choices=["GAIIx", "HiSeq2000", "HiSeq2500", "XTen"])
    ap.add_argument("--opts", action="append", default=None, help="one run with these ssc_set_option settings (repeatable)")
    ap.add_argument("--workdir", default=os.environ.get("SIMUSCOP_BENCH_DIR", "/tmp/simuscop_bench"))
    ap.add_argument("--trace-dir", default="", help="keep the chrome traces here (default: a temporary directory)")
    a = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    import bench
    import __graft_entry__ as ge
    from simuscop_b200 import cuda_binding, host_binding
    ge.build()
    os.makedirs(a.workdir, exist_ok=True)
    cfg, _ = bench.write_job(a.workdir, a.genome_bases, a.coverage, a.profile)
    job = host_binding.Job(cfg, 1)
    torch.cuda.init()
    gen = cuda_binding.Generator(0)
    gen.set_option("batch_pairs", a.batch_pairs)
    planned, _ = job.prepare(0, gen)
    bp = a.batch_pairs
    nbatch = planned // bp
    if max(a.warmup, a.batches) > nbatch:
        raise SystemExit("the job has %d batches of %d pairs" % (nbatch, bp))
    print("card: %s" % card(), flush=True)
    trace_dir = a.trace_dir or tempfile.mkdtemp(prefix="pipeline_probe_")
    os.makedirs(trace_dir, exist_ok=True)
    first = 0

    def span(n):
        """the next n batches of the job, wrapping to its start: every call reads and writes what no recent call touched"""
        nonlocal first
        if first + n > nbatch:
            first = 0
        first += n
        return (first - n) * bp, first * bp

    for run, opts in enumerate(a.opts or [""]):
        for kv in filter(None, opts.split(",")):
            gen.set_option(kv.split("=")[0], int(kv.split("=")[1]))
        gen.generate_device(*span(a.warmup))
        gen.reset_stats()
        plain = gen.generate_device(*span(a.batches))
        gen.reset_stats()
        rg = span(a.batches)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            res = gen.generate_device(*rg)
            torch.cuda.synchronize()
        st = gen.stats()
        path = os.path.join(trace_dir, "pipeline_probe_%d.json" % run)
        prof.export_chrome_trace(path)
        with open(path) as f:
            rows = per_batch(kernel_events(json.load(f)))
        print("opts %r: %d batches of %d pairs" % (opts, a.batches, bp))
        print("%5s %7s %7s %7s %7s %-8s %7s %7s %7s" % ("batch", "setup", "wait", "gen", "scan", "stream", "move", "step", "slack"))
        fmt = lambda r, k: "%7.3f" % r[k] if k in r else "%7s" % "-"    # noqa: E731
        for r in rows:
            print("%5d %s %s %s %s %-8s %s %s %s" % (r["batch"], fmt(r, "setup"), fmt(r, "wait"), fmt(r, "gen"), fmt(r, "scan"),
                                                     r.get("scan_stream", "-"), fmt(r, "move"), fmt(r, "step"), fmt(r, "slack")))
        nb = max(1, st["timed_batches"])
        s = {"opts": opts, "profile": a.profile, "median_ms": summary(rows),
             "stats_ms": {"gen": st["gen_kernel_ms"] / nb, "pass2": st["compact_kernel_ms"] / nb,
                          "mover": st["mover_kernel_ms"] / max(1, nb - 1) if "mover_kernel_ms" in st else "not measured",
                          "step": res["device_ms"] / a.batches},
             "unprofiled_step_ms": plain["device_ms"] / a.batches}
        print(json.dumps(s), flush=True)
    if not a.trace_dir:
        for p in glob.glob(os.path.join(trace_dir, "*.json")):
            os.remove(p)
        os.rmdir(trace_dir)
    gen.close()
    job.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
