"""Interleaved paired-end output (ssc_set_option "interleave", SIMUSCOP_INTERLEAVE, SIMUSCOP_STDOUT): one stream holding pair i
mate 1, pair i mate 2, ... in pair order, for `bwa mem -p` / `bowtie2 --interleaved` on standard input.

Every check compares the stream with the interleave of the _1 / _2 output of the same handle (or of the oracle, which the parity
suites pin to the reference): on the parity scenarios, on every fast-kernel instance at the read-length edges with and without
no_splice, on the generic and FP64 kernels, with batch / grid / mover options, over arbitrary pair ranges and shards, on the
hand-built plans of test_gpu_plan_edges (64-byte names of every byte value, 10-digit fields, pair IDs past 2^32), in gzip mode
member by member against the host mirror, at 2 M pairs per plan with the batch clamp, for array output, and through the CLI."""
import gzip
import os
import subprocess
import time

import numpy as np
import pytest

import helpers
from simuscop_b200 import planfile
from test_gpu_kernel_matrix import (EDGE, FAST, FP64, GENERIC_GLOBAL, GENERIC_SMEM, QMODES, check_path,  # noqa: F401
                                    fast_nch, reference)
from test_gpu_output_side import STORED_EXTRA, bases, expanding_cases, host_member, split_members  # noqa: F401 (fixtures)
from test_gpu_plan_edges import SEED, TICKET, Builder, cases, huge_bins, load, profiles, random_genome  # noqa: F401 (fixtures)

pytestmark = pytest.mark.gpu


def interleave(f1, f2):
    """(the interleave of the records of a _1 / _2 file pair, byte offset of every pair in it and the end).  The headers of a
    pair's two records agree but for the mate digit, which finds the header's end whatever bytes the name holds; the base line
    holds no line feed, and the quality line is as long as it."""
    out, offs = [], [0]
    p1 = p2 = 0
    while p1 < len(f1):
        k = len(os.path.commonprefix([f1[p1:p1 + 100], f2[p2:p2 + 100]]))
        assert f1[p1 + k:p1 + k + 2] == b"1\n" and f2[p2 + k:p2 + k + 2] == b"2\n", (p1, p2)
        H = k + 2
        n1 = H + 2 * (f1.index(b"\n", p1 + H) - p1 - H) + 4
        n2 = H + 2 * (f2.index(b"\n", p2 + H) - p2 - H) + 4
        out += [f1[p1:p1 + n1], f2[p2:p2 + n2]]
        offs.append(offs[-1] + n1 + n2)
        p1 += n1
        p2 += n2
    assert p2 == len(f2)
    return b"".join(out), offs


def expect(f1, f2):
    return interleave(f1, f2)[0] if f2 else f1


def check_handle(g, lo=0, hi=None):
    """On one handle: the two-file output of [lo, hi), then the interleaved one, equal to its interleave (SE: the same bytes),
    with the same statistics; ssc_generate_device returns the stream's length in bytes1 and 0 in bytes2.  Leaves the option off."""
    if hi is None:
        hi = g.planned
    g.set_option("interleave", 0)
    g.reset_stats()
    f1, f2 = g.generate(lo, hi)
    want = g.stats()
    g.set_option("interleave", 1)
    g.reset_stats()
    i1, i2 = g.generate(lo, hi)
    got = g.stats()
    exp = expect(f1, f2)
    assert i2 == b""
    assert helpers.first_diff(i1, exp) == -1, "interleaved stream differs at byte %d" % helpers.first_diff(i1, exp)
    for k in ("pairs_emitted", "reads_emitted", "bases_emitted", "fastq_bytes", "gz_bytes", "gen_kernel", "gen_nch", "gen_qmode"):
        assert got[k] == want[k], (k, got[k], want[k])
    d = g.generate_device(lo, hi)
    assert (d["bytes1"], d["bytes2"]) == (len(exp), 0), d
    g.set_option("interleave", 0)
    return f1, f2, i1


@pytest.fixture(scope="module")
def gen(built):
    from simuscop_b200 import cuda_binding
    g = cuda_binding.Generator(0)
    yield g
    g.close()


def scenario(name, workdir):
    scn = helpers.build_scenario(name, workdir)
    return planfile.read_plan(helpers.plan_dumps(scn, "ilv")[0]), scn


# ---------------------------------------------------------------------------------------------------------------------------
# 1. parity scenarios
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["pe_xten", "pe_tiny", "pe_variants", "pe_wes", "pe_ploidy3", "pe_iupac", "se_gaiix", "se_tumor"])
def test_parity_scenarios(name, gen, workdir):
    """PE: the stream is the interleave of the same handle's two files (pe_tiny: also of the instrumented reference's files);
    SE: the option changes nothing."""
    plan, scn = scenario(name, workdir)
    gen.load_plan(plan, scn["seed"])
    f1, f2, i1 = check_handle(gen)
    assert bool(f2) == plan.paired and len(f1) > 0
    if name == "pe_tiny":
        plans, out = helpers.reference_run(scn, tag="ilv_ref")
        r1, r2 = (helpers.read_file(p) for p in helpers.sample_files(out, planfile.read_plan(plans[0]), 0, scn))
        assert i1 == interleave(r1, r2)[0]


# ---------------------------------------------------------------------------------------------------------------------------
# 2. every instance
# ---------------------------------------------------------------------------------------------------------------------------
def run_interleaved(plan, seed, **options):
    from simuscop_b200 import cuda_binding
    g = cuda_binding.Generator(0)
    try:
        for k, v in options.items():
            g.set_option(k, v)
        g.set_option("interleave", 1)
        g.load_plan(plan, seed)
        i1, i2 = g.generate()
        return i1, i2, g.stats()
    finally:
        g.close()


@pytest.mark.parametrize("rl,qmode,splice", [pytest.param(rl, q, s, id="rl%d-nch%d-qp%d%s" % (rl, fast_nch(rl), q, "" if s else "-nosplice"))
                                             for rl in EDGE for q in QMODES for s in (True, False)])
def test_fast_instances(rl, qmode, splice, reference, check_path):  # noqa: F811
    """Every (NCH, QP) instance of the interleaved fast kernel at the read-length edges, spliced and position-by-position indel
    reads, against the oracle's two files (SE profiles: the option has no effect)."""
    plan, seed, o1, o2 = reference("rl%d" % rl)
    i1, i2, st = run_interleaved(plan, seed, fast_qmode=qmode, no_splice=0 if splice else 1)
    assert i2 == b"" and helpers.first_diff(i1, expect(o1, o2)) == -1, helpers.first_diff(i1, expect(o1, o2))
    check_path(st, (FAST, fast_nch(rl), qmode))


GENERIC_RUNS = {
    "rl161_b20": ({}, (GENERIC_SMEM, 10, -1)),
    "rl256_b31": ({}, (GENERIC_SMEM, 10, -1)),
    "rl320_b76": ({}, (GENERIC_GLOBAL, 10, -1)),
    "k5_b3": ({}, (GENERIC_GLOBAL, 10, -1)),
    "k8_b2": ({}, (GENERIC_GLOBAL, 10, -1)),
    "rl160-force_generic": ({"force_generic": 1}, (GENERIC_SMEM, 10, -1)),
    "rl65-force_generic": ({"force_generic": 1}, (GENERIC_SMEM, 10, -1)),
    "rl160-fp64_search": ({"fp64_search": 1}, (FP64, 10, -1)),
    "rl320_b76-fp64_search": ({"fp64_search": 1}, (FP64, 10, -1)),
}


@pytest.mark.parametrize("name", GENERIC_RUNS)
def test_generic_instances(name, reference, check_path):  # noqa: F811
    """The generic kernel's three interleaved instances: RL 161 / 256 / 320, K = 5 and 8, tables in shared and in global memory,
    forced on fast-kernel profiles, and the FP64 linear search."""
    options, want = GENERIC_RUNS[name]
    plan, seed, o1, o2 = reference(name.split("-")[0])
    assert plan.paired
    i1, i2, st = run_interleaved(plan, seed, **options)
    assert i2 == b"" and helpers.first_diff(i1, expect(o1, o2)) == -1, helpers.first_diff(i1, expect(o1, o2))
    check_path(st, want)


# ---------------------------------------------------------------------------------------------------------------------------
# 3. pipeline and ranges
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("option", [("batch_pairs", 256), ("max_ctas", 1), ("concurrent_move", 0), ("concurrent_move", 9)])
def test_options(option, built, workdir):
    """Many batches, one CTA whose warps take many tickets, the stand-alone move after every batch and the bulk-copy mover."""
    from simuscop_b200 import cuda_binding
    plan, scn = scenario("pe_variants", workdir)
    g = cuda_binding.Generator(0)
    try:
        g.set_option(*option)
        g.load_plan(plan, scn["seed"])
        if option[0] == "batch_pairs":
            assert g.emitted > 4 * 256
        check_handle(g)
    finally:
        g.close()


def test_ranges_and_shards(built, workdir):
    """Arbitrary [lo, hi), empty ones included; two handles on two shards concatenate to the one-handle stream; the option is
    switched on and off between calls on one handle."""
    from simuscop_b200 import cuda_binding
    plan, scn = scenario("pe_variants", workdir)
    g = cuda_binding.Generator(0)
    g2 = cuda_binding.Generator(0)
    try:
        g.set_option("batch_pairs", 512)
        g.load_plan(plan, scn["seed"])
        _, _, whole = check_handle(g)
        rng = np.random.default_rng(9)
        for lo, hi in [(0, 1), (0, 0), (7, 7), (g.planned, g.planned), (g.planned - 1, g.planned)] + \
                [tuple(sorted(int(x) for x in rng.integers(0, g.planned + 1, 2))) for _ in range(6)]:
            f1, f2, i1 = check_handle(g, lo, hi)
            if lo == hi:
                assert i1 == b"" and f1 == b""
        g2.set_option("interleave", 1)
        g2.load_plan(plan, scn["seed"])
        mid = g.planned // 2 + 3
        g.set_option("interleave", 1)
        assert g.generate(0, mid)[0] + g2.generate(mid, g.planned)[0] == whole
    finally:
        g.close()
        g2.close()


@pytest.mark.parametrize("mode", ["fast", "gzip", "generic"])
@pytest.mark.parametrize("name", ["names", "twin", "pair_ids"])
def test_plan_edges(name, mode, cases):  # noqa: F811
    """Names of 1..64 bytes with every byte value (line feeds too), fragment counters of 1..10 digits, pair IDs across 2^31,
    2^32 and 2^33 inside a ticket: the oracle's pair ranges of test_gpu_plan_edges; gzip output inflates to the same stream."""
    from simuscop_b200 import cuda_binding
    case = cases(name, "pe")
    g = cuda_binding.Generator(0)
    try:
        g.set_option("interleave", 1)
        if mode == "gzip":
            g.set_option("gzip", 1)
        if mode == "generic":
            g.set_option("force_generic", 1)
        load(g, case)
        for lo, hi, o1, o2 in case["jobs"]:
            i1, i2 = g.generate(lo, hi)
            if mode == "gzip":
                i1 = gzip.decompress(i1)
            exp = expect(o1, o2)
            assert i2 == b"" and helpers.first_diff(i1, exp) == -1, (lo, hi, helpers.first_diff(i1, exp))
    finally:
        g.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 4. gzip
# ---------------------------------------------------------------------------------------------------------------------------
def check_gzip_members(g, f1, f2, batch):
    """gzip + interleave on handle g (plan loaded, whole plan in batches of `batch` pairs): inflates to the interleave of f1 / f2,
    one member per ticket of both mates, each at most raw + 23 bytes and equal to the host mirror's member of the same blob with
    the table fitted to the first min(256, tickets of the first batch) tickets.  Returns (the stream, statistics, members)."""
    stream, offs = interleave(f1, f2)
    g.set_option("interleave", 1)
    g.set_option("gzip", 1)
    z1, z2 = g.generate()
    st = g.stats()
    assert z2 == b"" and gzip.decompress(z1) == stream
    n = len(offs) - 1
    sample = stream[:offs[min(n, batch, 256 * TICKET)]]
    tickets = [(t, min(b + batch, n, t + TICKET)) for b in range(0, n, batch) for t in range(b, min(b + batch, n), TICKET)]
    members = split_members(z1)
    assert len(members) == len(tickets), (len(members), len(tickets))
    for j, ((a, b), m) in enumerate(zip(tickets, members)):
        blob = stream[offs[a]:offs[b]]
        assert len(m) <= len(blob) + STORED_EXTRA and m == host_member(blob, sample), "member %d of %d bytes (blob %d)" % (j, len(m), len(blob))
    return z1, st, members


@pytest.mark.parametrize("batch", [0, 4096])
def test_gzip_members(batch, built, workdir):
    """XTen, default batches and batches of 4096 pairs: members of both mates, equal to ssc_gzip_member_host's; fastq_bytes /
    gz_bytes as in two-file gzip mode."""
    from simuscop_b200 import cuda_binding
    plan, scn = scenario("pe_xten", workdir)
    g = cuda_binding.Generator(0)
    try:
        if batch:
            g.set_option("batch_pairs", batch)
        g.load_plan(plan, scn["seed"])
        f1, f2 = g.generate()
        g.set_option("gzip", 1)
        g.reset_stats()
        z1, z2 = g.generate()
        two = g.stats()
        g.reset_stats()
        z, st, _ = check_gzip_members(g, f1, f2, batch or 1 << 20)
        assert st["fastq_bytes"] == two["fastq_bytes"] == len(f1) + len(f2)
        assert st["gz_bytes"] == len(z) and two["gz_bytes"] == len(z1) + len(z2)
        assert gzip.decompress(z1) == f1 and gzip.decompress(z2) == f2
    finally:
        g.close()


def test_gzip_stored_members(expanding_cases):  # noqa: F811
    """256 tickets of ACGT reads, then 64 of reads in an N run with 64-byte names of bytes the table was not fitted to: those
    members are stored, one block of raw + 23 bytes (raw: 32 records of both mates, below 65 535 bytes)."""
    from simuscop_b200 import cuda_binding
    case = expanding_cases("xten")
    o1, o2 = case["o"]
    g = cuda_binding.Generator(0)
    try:
        load(g, case)
        _, _, members = check_gzip_members(g, o1, o2, 1 << 20)
        stored = [m for m in members if (m[10] >> 1) & 3 == 0]
        assert len(stored) >= 64 and all(m[10] == 1 for m in stored)
        assert max(len(m) for m in stored) > 20480 + STORED_EXTRA      # longer than a two-file blob could be
    finally:
        g.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 5. batch clamp
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rl,batch", [(151, 0), (151, 1 << 21), (320, 0), (320, 1 << 21)])
def test_two_million_pairs(rl, batch, profiles, reference):  # noqa: F811
    """Plans of 2 097 152 pairs at RL 151 (fast kernel) and RL 320 (generic kernel), at the default batch size and at 2 M pairs per
    batch (clamped so that a slab of both mates stays below 2^31 bytes): no SSC_ERR_OVERFLOW, the stream is as long as the two
    files, and slices at the start, across the first batch boundaries and at the end equal their interleave."""
    from simuscop_b200 import cuda_binding
    base = profiles["pe"] if rl == 151 else reference("rl320_b76")[0]
    assert base.hdr["read_length"] == rl and base.paired
    genome = random_genome(20000, seed=3)
    b = Builder(True)
    b.segment(b"@ilv#chr1#", huge_bins(2 << 20, True, genome.size))
    plan = b.plan(base, genome)
    g = cuda_binding.Generator(0)
    try:
        if batch:
            g.set_option("batch_pairs", batch)
        g.load_plan(plan, SEED)
        assert g.emitted >= 2 << 20
        two = g.generate_device()
        g.set_option("interleave", 1)
        one = g.generate_device()
        assert (one["bytes1"], one["bytes2"]) == (two["bytes1"] + two["bytes2"], 0)
        n = g.planned
        for lo in (0, (1 << 20) - 700, 1 << 20, (1 << 21) - 2000, n - 3000):
            hi = min(n, lo + 3000)
            g.set_option("interleave", 0)
            f1, f2 = g.generate(lo, hi)
            g.set_option("interleave", 1)
            assert g.generate(lo, hi) == (interleave(f1, f2)[0], b"")
    finally:
        g.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 6. array output
# ---------------------------------------------------------------------------------------------------------------------------
def test_array_output_ignores_the_option(gen, workdir):
    import torch
    plan, scn = scenario("pe_variants", workdir)
    gen.load_plan(plan, scn["seed"])
    gen.set_option("interleave", 0)
    want = gen.generate_reads()
    want = {k: v.clone() for k, v in want.items()}
    gen.set_option("interleave", 1)
    got = gen.generate_reads()
    gen.set_option("interleave", 0)
    for k in ("reads", "length", "pair_id", "segment", "pos", "frag"):
        assert torch.equal(got[k], want[k]), k


# ---------------------------------------------------------------------------------------------------------------------------
# 7. CLI
# ---------------------------------------------------------------------------------------------------------------------------
def cli(scn, tag, **env_extra):
    """simuReads on scn's configuration with output directory out_<tag>; returns (CompletedProcess with bytes, output dir)."""
    from simuscop_b200 import paths, synth
    d = scn["dir"]
    out = os.path.join(d, "out_" + tag)
    cfg = os.path.join(d, "cfg_%s.txt" % tag)
    synth.write_config(cfg, output=out, **scn["kw"])
    env = dict(os.environ, SIMUSCOP_SEED=str(scn["seed"]), **env_extra)
    r = subprocess.run([paths.SIMUREADS, cfg], env=env, capture_output=True, timeout=600)
    return r, out


def test_cli_interleaved_files(built, workdir):
    """SIMUSCOP_INTERLEAVE=1 writes <stem>.fq (.fq.gz with SIMUSCOP_GZIP=1), the interleave of a normal run's _1 / _2 and no _1 / _2
    files, with one handle and with three (SIMUSCOP_DEVICES, 8192 pairs per batch)."""
    import torch
    scn = helpers.build_scenario("pe_tiny", workdir)
    r, out = cli(scn, "ilv_plain")
    assert r.returncode == 0, r.stderr[-3000:]
    want = interleave(helpers.read_file(os.path.join(out, "test_1.fq")), helpers.read_file(os.path.join(out, "test_2.fq")))[0]
    devs = "0,1,0" if torch.cuda.device_count() >= 2 else "0,0,0"
    for tag, env, fn in (("ilv", {}, "test.fq"), ("ilv_gz", {"SIMUSCOP_GZIP": "1"}, "test.fq.gz"),
                         ("ilv_three", {"SIMUSCOP_DEVICES": devs, "SIMUSCOP_BATCH_PAIRS": "8192"}, "test.fq"),
                         ("ilv_three_gz", {"SIMUSCOP_DEVICES": devs, "SIMUSCOP_BATCH_PAIRS": "8192", "SIMUSCOP_GZIP": "1"}, "test.fq.gz")):
        r, o = cli(scn, tag, SIMUSCOP_INTERLEAVE="1", **env)
        assert r.returncode == 0, (tag, r.stderr[-3000:])
        assert sorted(os.listdir(o)) == [fn], (tag, os.listdir(o))
        data = helpers.read_file(os.path.join(o, fn))
        assert (gzip.decompress(data) if fn.endswith(".gz") else data) == want, tag


def test_cli_stdout(built, workdir):
    """SIMUSCOP_STDOUT=1: standard output carries the interleaved FASTQ and nothing else, the messages go to stderr, no FASTQ file
    is created, the truth VCF still is; an SE configuration gives its <stem>.fq bytes; gzip is honoured."""
    scn = helpers.build_scenario("pe_tiny", workdir)
    r, out = cli(scn, "so_file", SIMUSCOP_INTERLEAVE="1")
    assert r.returncode == 0
    want = helpers.read_file(os.path.join(out, "test.fq"))
    r, out = cli(scn, "so", SIMUSCOP_STDOUT="1", SIMUSCOP_TRUTH_VCF="1")
    assert r.returncode == 0, r.stderr[-3000:]
    assert r.stdout == want and b"Reads generation done!" in r.stderr
    assert sorted(os.listdir(out)) == ["test.truth.vcf"]
    r, out = cli(scn, "so_gz", SIMUSCOP_STDOUT="1", SIMUSCOP_GZIP="1")
    assert r.returncode == 0 and gzip.decompress(r.stdout) == want and os.listdir(out) == []
    se = helpers.build_scenario("se_gaiix", workdir)
    r, out = cli(se, "so_se_file")
    assert r.returncode == 0
    want = helpers.read_file(os.path.join(out, "test.fq"))
    r, out = cli(se, "so_se", SIMUSCOP_STDOUT="1")
    assert r.returncode == 0 and r.stdout == want and os.listdir(out) == []


def test_cli_stdout_refuses_several_samples(built, workdir):
    """A tumour configuration with two abundance rows yields two samples: refused with exit 1 and a message, nothing generated."""
    scn = helpers.build_scenario("se_tumor", workdir)
    r, out = cli(scn, "so_two", SIMUSCOP_STDOUT="1")
    assert r.returncode == 1 and r.stdout == b""
    assert b"SIMUSCOP_STDOUT" in r.stderr and b"Reads generation done!" not in r.stderr
    assert not os.path.exists(out) or os.listdir(out) == []


def test_cli_stdout_reader_closes_early(built, workdir):
    """The reader takes the first kilobyte and closes the pipe: the CLI ends with a non-zero exit and an error message instead
    of hanging, and no process is left."""
    from simuscop_b200 import paths, synth
    scn = helpers.build_scenario("pe_xten", workdir)
    d = scn["dir"]
    cfg = os.path.join(d, "cfg_so_close.txt")
    synth.write_config(cfg, output=os.path.join(d, "out_so_close"), **scn["kw"])
    env = dict(os.environ, SIMUSCOP_SEED=str(scn["seed"]), SIMUSCOP_STDOUT="1")
    p = subprocess.Popen([paths.SIMUREADS, cfg], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    try:
        head = p.stdout.read(1024)
        assert len(head) == 1024 and head.startswith(b"@")
        p.stdout.close()
        t0 = time.time()
        _, err = p.communicate(timeout=120)
        assert p.returncode != 0 and b"Error" in err, (p.returncode, err[-2000:])
        assert time.time() - t0 < 120
    finally:
        if p.poll() is None:
            p.kill()
            p.wait()
