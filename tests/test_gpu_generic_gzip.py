"""gzip and BGZF output from the generic generation kernel (generate_kernel<K3, FP64, ILV, BLOB = true>): the profiles the fast
kernel does not take (RL 161..320, K != 3, tables too large for shared memory) and the FP64 search.

In gzip mode the generic kernel writes each tile of 32 pairs as one ticket blob per file, the same tickets the fast kernel cuts,
and the deflate kernel and pass 2 turn them into members.  Every run goes through test_gpu_bgzf's check_range (plain, gzip and
gzip + bgzf on one handle; the blocks walked, inflated to whole records, equal to the gzip members with the BC field, paired
across mates, the statistics and ssc_generate_device's lengths), and every block is compared with ssc_gzip_member_host's
member of its 32-pair blob, with the table fitted to the first min(256, tickets of the first batch) tickets.  On fast-kernel
plans the generic and FP64 kernels give the fast kernel's compressed bytes exactly."""
import gzip
import os
import shutil
import subprocess

import pytest

import helpers
from simuscop_b200 import planfile, synth
from test_gpu_bgzf import check_file, check_range, headers, inflate, to_bgzf, walk
from test_gpu_interleave import cli, interleave
from test_gpu_kernel_matrix import FAST, FP64, GENERIC_GLOBAL, GENERIC_SMEM, check_path, reference  # noqa: F401 (fixtures)
from test_gpu_output_side import expanding_cases, host_member, split_members  # noqa: F401 (fixtures)
from test_gpu_plan_edges import TICKET, load, profiles, records  # noqa: F401 (fixtures)

pytestmark = pytest.mark.gpu

DEFAULT_BATCH = 1 << 20
FAST_LARGEST_BLOCK = 39168 + 31          # an interleaved ticket of the fast kernel (RL <= 160) as a stored BGZF block

# generic-only plans (test_gpu_kernel_matrix.CASES, and the K = 4 stress profile) -> the instance that runs them
GENERIC_PLANS = {"rl161_b20": (GENERIC_SMEM, 10, -1), "rl256_b31": (GENERIC_SMEM, 10, -1), "rl320_b45": (GENERIC_SMEM, 10, -1),
                 "rl320_b76": (GENERIC_GLOBAL, 10, -1), "k5_b3": (GENERIC_GLOBAL, 10, -1), "k8_b2": (GENERIC_GLOBAL, 10, -1),
                 "k4_long": (GENERIC_GLOBAL, 10, -1)}


@pytest.fixture(scope="module")
def plans(reference, workdir):
    """name -> (plan, seed, oracle FASTQ 1, oracle FASTQ 2): the kernel-matrix cases, and helpers.STRESS["k4_long"]."""
    from oracle import binding as oracle_binding
    cache = {}

    def get(name):
        if name not in cache:
            if name in helpers.STRESS:
                scn = helpers.build_stress(name, workdir)
                plan = planfile.read_plan(helpers.plan_dumps(scn, "ggz")[0])
                cache[name] = (plan, scn["seed"]) + oracle_binding.generate(plan, scn["seed"])[:2]
            else:
                cache[name] = reference(name)
        return cache[name]
    return get


def streams(plan, o1, o2, ilv):
    """[(bytes, byte offset of every pair's records and the end)] of each output stream of the oracle's files."""
    if ilv and plan.paired:
        return [interleave(o1, o2)]
    return [(o1, records(o1))] + ([(o2, records(o2))] if plan.paired else [])


def check_blocks(blocks, strm, batch):
    """Block j of each stream is ssc_gzip_member_host's member of ticket j's blob as a BGZF block, the table fitted to the first
    min(256, tickets of the first batch) tickets of every stream; the batches of the library cut the tickets."""
    n = len(strm[0][1]) - 1
    B = -(-min(batch, n) // TICKET) * TICKET
    tickets = [(t, min(b + B, n, t + TICKET)) for b in range(0, n, B) for t in range(b, min(b + B, n), TICKET)]
    s_hi = min(n, B, 256 * TICKET)
    sample = b"".join(s[:offs[s_hi]] for s, offs in strm)
    assert len(blocks) == len(strm)
    for f, ((s, offs), bl) in enumerate(zip(strm, blocks)):
        assert len(bl) == len(tickets), (f, len(bl), len(tickets))
        for j, ((a, b), blk) in enumerate(zip(tickets, bl)):
            assert blk == to_bgzf(host_member(s[offs[a]:offs[b]], sample)), "stream %d, block %d of %d bytes" % (f + 1, j, len(blk))


def run_checked(plan, seed, o1, o2, options, load_case=None):
    """check_range over the whole plan on a new handle with `options`, then every block against the host mirror.  Returns
    (blocks per stream, statistics)."""
    from simuscop_b200 import cuda_binding
    ilv = bool(options.get("interleave")) and plan.paired
    g = cuda_binding.Generator(0)
    try:
        for k, v in options.items():
            g.set_option(k, v)
        if load_case is None:
            g.load_plan(plan, seed)
        else:
            load(g, load_case)
        _, blocks = check_range(g, want=(interleave(o1, o2)[0], b"") if ilv else (o1, o2))
        st = g.stats()
        check_blocks(blocks, streams(plan, o1, o2, ilv), options.get("batch_pairs", DEFAULT_BATCH))
        return blocks, st
    finally:
        g.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 1. generic-only plans
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batch", [0, 256])
@pytest.mark.parametrize("layout", ["two_file", "interleaved"])
@pytest.mark.parametrize("name", GENERIC_PLANS)
def test_generic_plans(name, layout, batch, plans, check_path):  # noqa: F811
    """Every generic instance in gzip and BGZF mode, two-file and interleaved (SE: the option has no effect), at the default
    batch size and at 256 pairs per batch: the oracle's bytes, members equal to the host mirror's, BGZF blocks within 64 KiB
    holding whole records (the same pairs in both files), the byte statistics, and the instance that ran."""
    plan, seed, o1, o2 = plans(name)
    options = {"interleave": 1} if layout == "interleaved" else {}
    if batch:
        options["batch_pairs"] = batch
    blocks, st = run_checked(plan, seed, o1, o2, options)
    check_path(st, GENERIC_PLANS[name])
    if batch:
        assert len(records(o1)) - 1 > batch          # several batches


# ---------------------------------------------------------------------------------------------------------------------------
# 2. the fast kernel's bytes
# ---------------------------------------------------------------------------------------------------------------------------
def compressed(plan, seed, options):
    """gzip and BGZF output, two-file and interleaved, of one handle with `options` (set before the plan): {(interleave, bgzf):
    (stream 1, stream 2)} and the instance that ran."""
    from simuscop_b200 import cuda_binding
    g = cuda_binding.Generator(0)
    try:
        for k, v in options.items():
            g.set_option(k, v)
        g.load_plan(plan, seed)
        g.set_option("gzip", 1)
        out = {}
        for ilv in (0, 1):
            for bgzf in (0, 1):
                g.set_option("interleave", ilv)
                g.set_option("bgzf", bgzf)
                out[(ilv, bgzf)] = g.generate()
        return out, g.stats()["gen_kernel"]
    finally:
        g.close()


@pytest.mark.parametrize("batch", [0, 256])
@pytest.mark.parametrize("name", ["rl65", "rl160", "pe_variants"])
def test_same_bytes_as_the_fast_kernel(name, batch, plans, workdir):
    """On plans the fast kernel takes, force_generic and fp64_search give the fast kernel's .gz and BGZF bytes exactly, two-file
    and interleaved: the members cut the same 32-pair tickets and the table is fitted to the same bytes."""
    if name == "pe_variants":
        scn = helpers.build_scenario(name, workdir)
        plan, seed = planfile.read_plan(helpers.plan_dumps(scn, "ggz")[0]), scn["seed"]
    else:
        plan, seed = plans(name)[:2]
    base = {"batch_pairs": batch} if batch else {}
    want, kernel = compressed(plan, seed, base)
    assert kernel == FAST
    assert all(want[(0, b)][1] for b in (0, 1)) and all(want[(1, b)][1] == b"" for b in (0, 1))
    for opt, kernels in (("force_generic", (GENERIC_SMEM, GENERIC_GLOBAL)), ("fp64_search", (FP64,))):
        got, kernel = compressed(plan, seed, dict(base, **{opt: 1}))
        assert kernel in kernels, (opt, kernel)
        for k in want:
            assert got[k] == want[k], (opt, k, [len(x) for x in got[k]], [len(x) for x in want[k]])


# ---------------------------------------------------------------------------------------------------------------------------
# 3. stored blocks past the fast kernel's largest
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def bases(built, workdir):
    """The base plan expanding_cases builds on: PE at RL 320 (generic kernel), inserts of at least the read length (no bin is
    risky: emitted == planned)."""
    d = os.path.join(workdir, "generic_gzip_base")
    os.makedirs(d, exist_ok=True)
    ref = os.path.join(d, "ref.fa")
    synth.make_genome(ref, [5000], seed=31)
    prof = os.path.join(d, "synthetic.profile")
    synth.write_profile(prof, seed=320, kmer=3, read_length=320, bins=45, n_live_qual=7)
    kw = dict(ref=ref, profile=prof, layout="PE", coverage=1, insertSize=480, threads=1, verbose=0, name="p")
    b = planfile.read_plan(helpers.plan_dumps(dict(dir=d, kw=kw, seed=1, name="generic_gzip_base"), "p")[0])
    assert b.hdr["read_length"] == 320 and b.hdr["kmer"] == 3 and b.hdr["min_insert_size"] >= 320
    return {"rl320": b}


def test_stored_blocks_past_the_fast_kernel(expanding_cases):  # noqa: F811
    """256 tickets of ACGT reads, then 64 tickets in an N run whose 64-byte names carry bytes the table was not fitted to, at
    RL 320, interleaved: those tickets are stored blocks of raw + 31 bytes, longer than any block of the fast kernel, below
    64 KiB, each one well-formed stored block equal to the host mirror's."""
    case = expanding_cases("rl320")
    o1, o2 = case["o"]
    blocks, _ = run_checked(case["plan"], None, o1, o2, {"interleave": 1}, load_case=case)
    stored = [b for b in blocks[0] if (b[18] >> 1) & 3 == 0]
    assert len(stored) >= 64
    assert max(len(b) for b in stored) > FAST_LARGEST_BLOCK
    for b in stored:
        n = len(b) - 31
        assert b[18] == 1 and b[19:23] == bytes([n & 255, n >> 8, ~n & 255, (~n >> 8) & 255]) and len(b) <= 65536
        headers(inflate(b))


# ---------------------------------------------------------------------------------------------------------------------------
# 4. CLI
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def rl250(built, workdir):
    """A configuration with a synthetic K = 3 PE profile at RL 250 (the generic kernel)."""
    d = os.path.join(workdir, "generic_gzip_rl250")
    os.makedirs(d, exist_ok=True)
    ref = os.path.join(d, "ref.fa")
    synth.make_genome(ref, [200000, 30000], seed=41, n_runs=2, lower_runs=1, run_len=300)
    prof = os.path.join(d, "synthetic.profile")
    synth.write_profile(prof, seed=250, kmer=3, read_length=250, bins=31, n_live_qual=12)
    kw = dict(ref=ref, profile=prof, layout="PE", coverage=6, insertSize=340, threads=1, verbose=0, name="test")
    return dict(dir=d, kw=kw, seed=9, name="generic_gzip_rl250")


def test_cli_bgzf_files(rl250):
    """SIMUSCOP_BGZF=1 on an RL 250 profile: _1 / _2 .fq.gz and their .gzi, inflating to the plain run's files, every index entry
    at a block that inflates to the bytes at its offset."""
    r, out = cli(rl250, "ggz_plain")
    assert r.returncode == 0, r.stderr[-3000:]
    plain = {f: helpers.read_file(os.path.join(out, f)) for f in os.listdir(out)}
    assert sorted(plain) == ["test_1.fq", "test_2.fq"]
    r, out = cli(rl250, "ggz_bgzf", SIMUSCOP_BGZF="1")
    assert r.returncode == 0, r.stderr[-3000:]
    assert sorted(os.listdir(out)) == ["test_1.fq.gz", "test_1.fq.gz.gzi", "test_2.fq.gz", "test_2.fq.gz.gzi"]
    for f, p in plain.items():
        data = helpers.read_file(os.path.join(out, f + ".gz"))
        check_file(data, p, helpers.read_file(os.path.join(out, f + ".gz.gzi")))
        assert len(walk(data)) > 2


def test_cli_stdout_gzip(rl250):
    """SIMUSCOP_STDOUT=1 SIMUSCOP_GZIP=1 on an RL 250 profile: exit 0 and one gzip stream of the interleaved reads."""
    r, out = cli(rl250, "ggz_plain_so")
    assert r.returncode == 0, r.stderr[-3000:]
    want = interleave(helpers.read_file(os.path.join(out, "test_1.fq")), helpers.read_file(os.path.join(out, "test_2.fq")))[0]
    r, out = cli(rl250, "ggz_so", SIMUSCOP_STDOUT="1", SIMUSCOP_GZIP="1")
    assert r.returncode == 0, r.stderr[-3000:]
    assert len(split_members(r.stdout)) > 1 and gzip.decompress(r.stdout) == want
    assert not os.path.exists(out) or os.listdir(out) == []


@pytest.mark.skipif(not (shutil.which("bgzip") or shutil.which("samtools")), reason="bgzip / samtools not installed")
def test_htslib_reads_the_files(rl250):
    """Where htslib's tools are installed: bgzip -t and a parallel bgzip -d accept an RL 250 file, samtools fqidx indexes it."""
    r, out = cli(rl250, "ggz_hts_plain")
    assert r.returncode == 0
    plain = helpers.read_file(os.path.join(out, "test_1.fq"))
    r, out = cli(rl250, "ggz_hts", SIMUSCOP_BGZF="1")
    assert r.returncode == 0
    path = os.path.join(out, "test_1.fq.gz")
    if shutil.which("bgzip"):
        assert subprocess.run(["bgzip", "-t", path], capture_output=True).returncode == 0
        d = subprocess.run(["bgzip", "-d", "-@4", "-c", path], capture_output=True)
        assert d.returncode == 0 and d.stdout == plain
    if shutil.which("samtools"):
        assert subprocess.run(["samtools", "fqidx", path], capture_output=True).returncode == 0
        rec = plain.split(b"\n")[40:44]
        name = rec[0][1:].split()[0].decode()
        q = subprocess.run(["samtools", "fqidx", path, name], capture_output=True)
        assert q.returncode == 0 and q.stdout.split(b"\n")[0].split()[0] == rec[0].split()[0]
