"""Unaligned BAM output (ssc_set_option "bam", ssc_set_read_group, ssc_bam_header, SIMUSCOP_BAM): BGZF blocks of BAM records
written by both generation kernels, one record per read, the reads and order of the interleaved FASTQ.

Every stream is decoded here (zlib + struct): each BGZF block is walked and inflated on its own to whole records (PE: whole
pairs, mate 1 then mate 2), every fixed field of every record is checked, and each record is turned back into its FASTQ
record -- '@' + name + "/1" or "/2" (PE) + bases + "+" + qualities + 33 -- which must give, byte for byte, the interleaved FASTQ
of the same handle and range, or of the oracle (which the parity suites pin to the reference)."""
import os
import shutil
import struct
import subprocess

import numpy as np
import pytest

import helpers
from simuscop_b200 import planfile
from test_gpu_bgzf import BGZF_EOF, inflate, walk
from test_gpu_generic_gzip import GENERIC_PLANS, plans  # noqa: F401 (fixtures)
from test_gpu_interleave import cli, expect
from test_gpu_kernel_matrix import EDGE, FAST, FP64, GENERIC_GLOBAL, GENERIC_SMEM, QMODES, check_path, fast_nch, reference  # noqa: F401
from test_gpu_plan_edges import NAME_BLOB_LIMIT, SEED, Builder, cases, load, oracle, profiles, random_genome  # noqa: F401

pytestmark = pytest.mark.gpu

NIBBLES = b"=ACMGRSVTWYHKDBN"
PAIR_CHARS = [bytes([NIBBLES[b >> 4], NIBBLES[b & 15]]) for b in range(256)]
FIXED = struct.Struct("<iiiBBHHHIiii")
assert FIXED.size == 36


def records(raw, rg):
    """The records of a run of whole BAM records, each checked field by field: [(flag, name, FASTQ bases, FASTQ qualities)]."""
    out, at = [], 0
    tag = b"RGZ" + rg + b"\0" if rg else b""
    while at < len(raw):
        bs, ref, pos, lrn, mapq, bin_, ncig, flag, lseq, nref, npos, tlen = FIXED.unpack_from(raw, at)
        assert (ref, pos, mapq, bin_, ncig, nref, npos, tlen) == (-1, -1, 0, 4680, 0, -1, -1, 0), (at, raw[at:at + 36].hex())
        assert flag in (77, 141, 4) and lrn >= 2
        nb = (lseq + 1) // 2
        assert bs + 4 == 36 + lrn + nb + lseq + len(tag), (at, bs, lrn, lseq)
        p = at + 36
        name = raw[p:p + lrn - 1]
        assert raw[p + lrn - 1] == 0 and b"\0" not in name
        p += lrn
        packed = raw[p:p + nb]
        if lseq & 1:
            assert packed[-1] & 15 == 0                                      # the pad nibble of an odd-length read
        seq = b"".join(PAIR_CHARS[b] for b in packed)[:lseq]
        p += nb
        qual = bytes(q + 33 for q in raw[p:p + lseq])
        p += lseq
        assert raw[p:p + len(tag)] == tag
        at = p + len(tag)
        out.append((flag, name, seq, qual))
    assert at == len(raw)
    return out


def to_fastq(recs):
    out = []
    for flag, name, seq, qual in recs:
        suffix = b"" if flag == 4 else (b"/1" if flag == 77 else b"/2")
        out.append(b"@" + name + suffix + b"\n" + seq + b"\n+\n" + qual + b"\n")
    return b"".join(out)


def decode(z, paired, rg):
    """(FASTQ of a stream of BGZF blocks of BAM records, raw BAM bytes): every block well-formed, whole records (PE: whole pairs
    with flags 77 / 141 and one name), a stored block raw + 31 bytes."""
    fq, nraw = [], 0
    for b in walk(z):
        raw = inflate(b)
        if (b[18] >> 1) & 3 == 0:
            assert b[18] == 1 and len(b) == len(raw) + 31
        recs = records(raw, rg)
        assert recs
        if paired:
            assert len(recs) % 2 == 0
            for r1, r2 in zip(recs[0::2], recs[1::2]):
                assert r1[0] == 77 and r2[0] == 141 and r1[1] == r2[1], (r1[:2], r2[:2])
        else:
            assert all(r[0] == 4 for r in recs)
        fq.append(to_fastq(recs))
        nraw += len(raw)
    return b"".join(fq), nraw


def bam_of(g, lo=0, hi=None, rg=None):
    """The BAM stream of pairs [lo, hi) on handle g: ((stream 1, stream 2), statistics of the call).  Leaves the option off."""
    g.set_read_group(rg)
    g.set_option("bam", 1)
    g.reset_stats()
    z = g.generate(lo, hi)
    st = g.stats()
    d = g.generate_device(lo, hi)
    assert (d["bytes1"], d["bytes2"]) == (len(z[0]), 0), d
    g.set_option("bam", 0)
    return z, st


def check_bam(g, want, lo=0, hi=None, rg=None, want_stats=None):
    """The BAM stream of [lo, hi) on g decodes to `want` (interleaved FASTQ), with the statistics of the FASTQ run."""
    paired = g.read_shape(0, 0)[1] == 2
    (z1, z2), st = bam_of(g, lo, hi, rg)
    assert z2 == b""
    fq, nraw = decode(z1, paired, rg.encode() if rg else b"")
    i = helpers.first_diff(fq, want)
    assert i == -1, "BAM differs from the interleaved FASTQ at byte %d of %d / %d" % (i, len(fq), len(want))
    assert st["gz_bytes"] == len(z1) and st["fastq_bytes"] == nraw
    if want_stats is not None:
        for k in ("pairs_emitted", "reads_emitted", "bases_emitted", "gen_kernel", "gen_nch", "gen_qmode"):
            assert st[k] == want_stats[k], (k, st[k], want_stats[k])
    return z1, st


def fastq_and_bam(g, lo=0, hi=None, rg=None):
    """On one handle: the interleaved FASTQ of [lo, hi), then its BAM, checked against it.  Returns (FASTQ, BAM, stats)."""
    g.set_option("bam", 0)
    g.set_option("interleave", 1)
    g.reset_stats()
    want = g.generate(lo, hi)[0]
    ws = g.stats()
    g.set_option("interleave", 0)
    z, st = check_bam(g, want, lo, hi, rg, ws)
    return want, z, st


@pytest.fixture(scope="module")
def gen(built):
    from simuscop_b200 import cuda_binding
    g = cuda_binding.Generator(0)
    yield g
    g.close()


def scenario(name, workdir):
    scn = helpers.build_scenario(name, workdir)
    return planfile.read_plan(helpers.plan_dumps(scn, "bam")[0]), scn


# ---------------------------------------------------------------------------------------------------------------------------
# 1. parity scenarios
# ---------------------------------------------------------------------------------------------------------------------------
PARITY = ["pe_xten", "pe_tiny", "pe_variants", "pe_wes", "pe_ploidy3", "pe_iupac", "se_gaiix", "se_tumor"]


@pytest.mark.parametrize("name", PARITY)
def test_parity_scenarios(name, gen, workdir):
    """The whole plan and a range inside tickets, with and without a read group; pe_tiny also against the oracle; pe_iupac holds
    N bases (code 15)."""
    plan, scn = scenario(name, workdir)
    gen.load_plan(plan, scn["seed"])
    want, z, st = fastq_and_bam(gen, rg="rg-" + name)
    assert st["gen_kernel"] == FAST
    if name == "pe_tiny":
        from oracle import binding as oracle_binding
        o1, o2, _ = oracle_binding.generate(plan, scn["seed"])
        assert want == expect(o1, o2)
    if name == "pe_iupac":
        assert b"N" in b"".join(want.split(b"\n")[1::4])
    fastq_and_bam(gen, 37, gen.planned - 45)


# ---------------------------------------------------------------------------------------------------------------------------
# 2. every instance
# ---------------------------------------------------------------------------------------------------------------------------
def run_bam(plan, seed, rg=None, **options):
    from simuscop_b200 import cuda_binding
    g = cuda_binding.Generator(0)
    try:
        for k, v in options.items():
            g.set_option(k, v)
        g.load_plan(plan, seed)
        g.set_read_group(rg)
        g.set_option("bam", 1)
        z = g.generate()
        return z, g.stats()
    finally:
        g.close()


@pytest.mark.parametrize("rl,qmode,splice", [pytest.param(rl, q, s, id="rl%d-nch%d-qp%d%s" % (rl, fast_nch(rl), q, "" if s else "-nosplice"))
                                             for rl in EDGE for q in QMODES for s in (True, False)])
def test_fast_instances(rl, qmode, splice, reference, check_path):  # noqa: F811
    """Every (NCH, QP) instance of the fast kernel in BAM mode at the read-length edges, odd and even lengths, spliced and
    position-by-position indel reads, against the oracle's interleaved records."""
    plan, seed, o1, o2 = reference("rl%d" % rl)
    rg = "edge%d" % rl if splice else None
    (z1, z2), st = run_bam(plan, seed, rg, fast_qmode=qmode, no_splice=0 if splice else 1)
    fq, nraw = decode(z1, plan.paired, rg.encode() if rg else b"")
    want = expect(o1, o2)
    assert z2 == b"" and helpers.first_diff(fq, want) == -1, helpers.first_diff(fq, want)
    assert st["fastq_bytes"] == nraw and st["gz_bytes"] == len(z1)
    check_path(st, (FAST, fast_nch(rl), qmode))


GENERIC_RUNS = dict({name: ({}, want) for name, want in GENERIC_PLANS.items()},
                    **{"rl161_b20-batch256": ({"batch_pairs": 256}, GENERIC_PLANS["rl161_b20"]),
                       "rl320_b76-batch256": ({"batch_pairs": 256}, GENERIC_PLANS["rl320_b76"]),
                       "rl160-fp64_search": ({"fp64_search": 1}, (FP64, 10, -1)),
                       "rl33-fp64_search": ({"fp64_search": 1}, (FP64, 10, -1)),
                       "rl320_b76-fp64_search": ({"fp64_search": 1}, (FP64, 10, -1)),
                       "rl97-force_generic": ({"force_generic": 1}, (GENERIC_SMEM, 10, -1))})


@pytest.mark.parametrize("name", GENERIC_RUNS)
def test_generic_instances(name, plans, check_path):  # noqa: F811
    """The generic kernel's BAM instances: RL 161 / 256 / 320, K = 4, 5 and 8, tables in shared and in global memory, PE and SE,
    256 pairs per batch, the FP64 search and force_generic, against the oracle."""
    options, want_path = GENERIC_RUNS[name]
    plan, seed, o1, o2 = plans(name.split("-")[0])
    (z1, z2), st = run_bam(plan, seed, "generic", **options)
    fq, nraw = decode(z1, plan.paired, b"generic")
    want = expect(o1, o2)
    assert z2 == b"" and helpers.first_diff(fq, want) == -1, helpers.first_diff(fq, want)
    assert st["fastq_bytes"] == nraw
    check_path(st, want_path)
    if "batch_pairs" in options:
        assert len(walk(z1)) > st["pairs_emitted"] // 256


# ---------------------------------------------------------------------------------------------------------------------------
# 3. pipeline options, switching formats, array output
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("option", [("batch_pairs", 256), ("max_ctas", 1), ("concurrent_move", 0), ("concurrent_move", 9)])
def test_options(option, built, workdir):
    from simuscop_b200 import cuda_binding
    plan, scn = scenario("pe_variants", workdir)
    g = cuda_binding.Generator(0)
    try:
        g.set_option(*option)
        g.load_plan(plan, scn["seed"])
        _, z, _ = fastq_and_bam(g, rg="opt")
        if option[0] == "batch_pairs":
            assert len(walk(z)) >= g.emitted // 256
    finally:
        g.close()


def test_switching_formats(built, workdir):
    """On one handle: FASTQ, gzip and BGZF, then BAM, then FASTQ, gzip and BGZF again, then BAM again.  Each format is the same
    as before the switch (the Huffman table is fitted anew for the format that runs), and BAM is a fresh handle's BAM."""
    from simuscop_b200 import cuda_binding
    plan, scn = scenario("pe_xten", workdir)

    def others(g):
        out = []
        for gz, bg in ((0, 0), (1, 0), (1, 1)):
            g.set_option("gzip", gz)
            g.set_option("bgzf", bg)
            out.append(g.generate())
        g.set_option("gzip", 0)
        g.set_option("bgzf", 0)
        return out

    fresh = cuda_binding.Generator(0)
    g = cuda_binding.Generator(0)
    try:
        fresh.load_plan(plan, scn["seed"])
        (want_bam, _), _ = bam_of(fresh, rg="x")
        g.load_plan(plan, scn["seed"])
        before = others(g)
        (b1, _), _ = bam_of(g, rg="x")
        assert b1 == want_bam
        assert others(g) == before
        # the other options do not change BAM output
        for k in ("gzip", "bgzf", "interleave"):
            g.set_option(k, 1)
        (b2, _), _ = bam_of(g, rg="x")
        assert b2 == want_bam
        for k in ("gzip", "bgzf", "interleave"):
            g.set_option(k, 0)
        assert others(g) == before
    finally:
        g.close()
        fresh.close()


def test_read_group_between_calls(gen, workdir):
    """The read group may change between calls, and be removed; a bad id is refused and leaves the last one."""
    from simuscop_b200 import cuda_binding
    plan, scn = scenario("pe_tiny", workdir)
    gen.load_plan(plan, scn["seed"])
    gen.set_option("interleave", 1)
    want = gen.generate()[0]
    gen.set_option("interleave", 0)
    for rg in ("a", "b" * 64, None, "", "~!x"):
        check_bam(gen, want, rg=rg)
    gen.set_read_group("kept")
    for bad in ("with space", "x" * 65, "\x7f"):
        with pytest.raises(cuda_binding.SscError):
            gen.set_read_group(bad)
    gen.set_option("bam", 1)
    z = gen.generate()[0]
    gen.set_option("bam", 0)
    assert decode(z, True, b"kept")[0] == want


def test_array_output_ignores_the_option(gen, workdir):
    import torch
    plan, scn = scenario("pe_variants", workdir)
    gen.load_plan(plan, scn["seed"])
    gen.set_option("bam", 0)
    want = {k: v.clone() for k, v in gen.generate_reads().items()}
    st0 = gen.stats()
    gen.set_option("bam", 1)
    got = gen.generate_reads()
    st1 = gen.stats()
    gen.set_option("bam", 0)
    for k in ("reads", "length", "pair_id", "segment", "pos", "frag"):
        assert torch.equal(got[k], want[k]), k
    assert st1["fastq_bytes"] == st0["fastq_bytes"] and st1["gz_bytes"] == st0["gz_bytes"]


# ---------------------------------------------------------------------------------------------------------------------------
# 4. hand-built plans
# ---------------------------------------------------------------------------------------------------------------------------
QNAME = bytes(c for c in range(0x21, 0x7f) if c != 0x40)


def qname_case(base):
    """Names of 1..64 bytes drawn from the QNAME alphabet [!-?A-~] after the '@' (every such byte occurs)."""
    RL = base.hdr["read_length"]
    n = 60000
    genome = random_genome(n, seed=43)
    b = Builder(base.paired)
    rng = np.random.default_rng(12)
    used = set()
    for L in list(range(1, 65)):
        nm = b"@" + bytes(QNAME[(7 * L + 3 * i) % len(QNAME)] for i in range(L - 1))
        used |= set(nm[1:])
        bins = []
        for _ in range(2):
            w = int(rng.integers(RL, 600))
            sp = int(rng.integers(0, n - 451 - RL - w))
            bins.append((0, n, sp, sp + w, int(rng.integers(500, 70000)), int(rng.integers(1, 4))))
        b.segment(nm, bins)
    assert used == set(QNAME)
    return b.plan(base, genome)


@pytest.fixture(scope="module")
def qnames(profiles):
    out = {}
    for layout in ("pe", "se"):
        plan = qname_case(profiles[layout])
        o1, o2, _ = oracle(plan)
        out[layout] = (plan, expect(o1, o2))
    return out


@pytest.mark.parametrize("mode", ["fast", "generic"])
@pytest.mark.parametrize("layout", ["pe", "se"])
def test_qname_alphabet(layout, mode, qnames):
    from simuscop_b200 import cuda_binding
    plan, want = qnames[layout]
    g = cuda_binding.Generator(0)
    try:
        if mode == "generic":
            g.set_option("force_generic", 1)
        g.load_plan(plan, SEED)
        check_bam(g, want, rg="names")
        assert g.stats()["gen_kernel"] == (FAST if mode == "fast" else GENERIC_SMEM)
    finally:
        g.close()


@pytest.mark.parametrize("mode", ["fast", "generic"])
@pytest.mark.parametrize("name", ["twin", "pair_ids"])
def test_plan_edges(name, mode, cases):  # noqa: F811
    """Fragment counters of 1..10 digits (names of up to 85 bytes) and pair IDs across 2^31, 2^32 and 2^33 inside a ticket."""
    from simuscop_b200 import cuda_binding
    case = cases(name, "pe")
    g = cuda_binding.Generator(0)
    try:
        if mode == "generic":
            g.set_option("force_generic", 1)
        load(g, case)
        for lo, hi, o1, o2 in case["jobs"]:
            check_bam(g, expect(o1, o2), lo, hi, rg="edges")
    finally:
        g.close()


def test_names_outside_the_qname_alphabet_are_refused(cases, qnames):
    """The every-byte names plan: SSC_ERR_INVALID naming the segment and the byte, before anything reaches the sink, from
    ssc_generate and ssc_generate_device; FASTQ output of the plan still works, and the handle then writes a valid plan's BAM."""
    from simuscop_b200 import cuda_binding
    case = cases("names", "pe")
    g = cuda_binding.Generator(0)
    try:
        load(g, case)
        g.set_option("bam", 1)
        called = []

        def sink(user, b1, l1, b2, l2, first, n):
            called.append(n)
            return 0
        with pytest.raises(cuda_binding.SscError) as e:
            g.generate(sink=sink)
        assert "segment 1:" in str(e.value) and "0x01" in str(e.value) and not called   # segment 0 is "@" alone
        with pytest.raises(cuda_binding.SscError):
            g.generate_device()
        g.set_option("bam", 0)
        lo, hi, o1, o2 = case["jobs"][0]
        assert g.generate(lo, hi) == (o1, o2)
        plan, want = qnames["pe"]
        g.load_plan(plan, SEED)
        check_bam(g, want)
    finally:
        g.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 5. CLI
# ---------------------------------------------------------------------------------------------------------------------------
def check_bam_file(data, want, paired, rg="test"):
    """A BAM file of the CLI: the header block of ssc_bam_header(rg), records decoding to `want` with RG:Z:<rg>, the EOF block
    (the read group is the sample's stem where it fits)."""
    from simuscop_b200 import cuda_binding
    hdr = cuda_binding.bam_header(rg)
    assert data.startswith(hdr) and data.endswith(BGZF_EOF)
    body = data[len(hdr):len(data) - len(BGZF_EOF)]
    fq, _ = decode(body, paired, rg.encode())
    assert helpers.first_diff(fq, want) == -1, helpers.first_diff(fq, want)


@pytest.mark.parametrize("key", ["pe_tiny", "se_gaiix"])
def test_cli_files(key, built, workdir):
    """SIMUSCOP_BAM=1: <stem>.bam and nothing else, equal in content to the SIMUSCOP_INTERLEAVE=1 run, also with the options it
    takes precedence over, and over three handles in batches of 256 pairs."""
    scn = helpers.build_scenario(key, workdir)
    paired = key.startswith("pe")
    r, out = cli(scn, "bam_fq_" + key, SIMUSCOP_INTERLEAVE="1")
    assert r.returncode == 0, r.stderr[-3000:]
    want = helpers.read_file(os.path.join(out, "test.fq"))
    runs = {"one": {}, "precedence": {"SIMUSCOP_GZIP": "1", "SIMUSCOP_BGZF": "1", "SIMUSCOP_INTERLEAVE": "1"},
            "three": {"SIMUSCOP_DEVICES": "0,0,0", "SIMUSCOP_BATCH_PAIRS": "256"}}
    files = {}
    for tag, env in runs.items():
        r, o = cli(scn, "bam_%s_%s" % (tag, key), SIMUSCOP_BAM="1", **env)
        assert r.returncode == 0, (tag, r.stderr[-3000:])
        assert sorted(os.listdir(o)) == ["test.bam"], (tag, os.listdir(o))
        files[tag] = helpers.read_file(os.path.join(o, "test.bam"))
        check_bam_file(files[tag], want, paired)
    assert files["precedence"] == files["one"]


def renamed(scn, old, new):
    """The scenario with every population name `old...` called `new...` (configuration and variation file)."""
    kw = dict(scn["kw"], name=scn["kw"]["name"].replace(old, new))
    if kw.get("variation"):
        path = os.path.join(scn["dir"], "variations_%s.txt" % new)
        with open(kw["variation"]) as f, open(path, "w") as g:
            g.write(f.read().replace("\t%s" % old, "\t%s" % new))
        kw["variation"] = path
    return dict(scn, kw=kw)


def test_cli_long_stems(built, workdir):
    """Two samples of a tumour mixture whose stems are longer than a read group id may be: each <stem>.bam carries the first 62
    bytes of its stem and "~<sample index>" as its read group, in the header and on every record."""
    scn = renamed(helpers.build_scenario("se_tumor", workdir), "clone", "clonal_population_")
    r, out = cli(scn, "bam_long_fq")
    assert r.returncode == 0, r.stderr[-3000:]
    fastq = sorted(f for f in os.listdir(out) if f.endswith(".fq"))
    assert len(fastq) == 2
    r, o = cli(scn, "bam_long", SIMUSCOP_BAM="1")
    assert r.returncode == 0, r.stderr[-3000:]
    assert sorted(os.listdir(o)) == sorted(f[:-3] + ".bam" for f in fastq)
    with open(scn["kw"]["abundance"]) as f:
        rows = [ln.split("\t") for ln in f.read().splitlines() if ln]
    names = scn["kw"]["name"].split(",")
    for i, row in enumerate(rows):
        stem = "+".join("%s_%.3f" % (n, float(p)) for n, p in zip(names, row))
        assert len(stem) > 64
        rg = stem[:62] + "~%d" % i
        want = helpers.read_file(os.path.join(out, stem + ".fq"))
        check_bam_file(helpers.read_file(os.path.join(o, stem + ".bam")), want, False, rg)


def test_cli_refuses_invalid_names_before_writing(built, workdir):
    """A population name holding '@' (not a BAM read-name character): exit 1 with the QNAME message, and no .bam file."""
    scn = renamed(helpers.build_scenario("pe_tiny", workdir), "test", "bad@name")
    r, out = cli(scn, "bam_badname", SIMUSCOP_BAM="1")
    assert r.returncode == 1 and b"QNAME" in r.stderr, r.stderr[-3000:]
    assert not any(f.endswith(".bam") for f in (os.listdir(out) if os.path.exists(out) else []))


def test_cli_two_gpus(built, workdir):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    scn = helpers.build_scenario("pe_tiny", workdir)
    r, out = cli(scn, "bam2_fq", SIMUSCOP_INTERLEAVE="1")
    assert r.returncode == 0
    want = helpers.read_file(os.path.join(out, "test.fq"))
    r, o = cli(scn, "bam2", SIMUSCOP_BAM="1", SIMUSCOP_DEVICES="0,1", SIMUSCOP_BATCH_PAIRS="256")
    assert r.returncode == 0, r.stderr[-3000:]
    check_bam_file(helpers.read_file(os.path.join(o, "test.bam")), want, True)


def test_cli_stdout(built, workdir):
    """SIMUSCOP_STDOUT=1 SIMUSCOP_BAM=1: the BAM stream on standard output, header block to EOF block, and no file."""
    scn = helpers.build_scenario("pe_tiny", workdir)
    r, out = cli(scn, "bam_so_fq", SIMUSCOP_STDOUT="1")
    assert r.returncode == 0
    want = r.stdout
    r, out = cli(scn, "bam_so", SIMUSCOP_STDOUT="1", SIMUSCOP_BAM="1")
    assert r.returncode == 0, r.stderr[-3000:]
    check_bam_file(r.stdout, want, True)
    assert not os.path.exists(out) or os.listdir(out) == []


@pytest.mark.skipif(not shutil.which("samtools"), reason="samtools not installed")
def test_samtools_reads_the_file(built, workdir):
    """Where samtools is installed: quickcheck passes and samtools fastq gives our records (names without /1 /2 suffixes)."""
    scn = helpers.build_scenario("pe_tiny", workdir)
    r, out = cli(scn, "bam_st_fq", SIMUSCOP_INTERLEAVE="1")
    assert r.returncode == 0
    want = helpers.read_file(os.path.join(out, "test.fq"))
    r, out = cli(scn, "bam_st", SIMUSCOP_BAM="1")
    assert r.returncode == 0
    path = os.path.join(out, "test.bam")
    assert subprocess.run(["samtools", "quickcheck", path], capture_output=True).returncode == 0
    q = subprocess.run(["samtools", "fastq", "-N", path], capture_output=True)
    assert q.returncode == 0 and q.stdout == want
