"""GPU parity: the CUDA path (through the C ABI) against the Philox-instrumented reference
and the C oracle, byte for byte."""
import pytest

import helpers
from simuscop_b200 import planfile

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gen(built):
    from simuscop_b200 import cuda_binding
    g = cuda_binding.Generator(0)
    yield g
    g.close()


@pytest.mark.parametrize("name", ["pe_xten", "se_gaiix", "pe_tiny", "pe_variants", "pe_wes", "se_tumor", "pe_ploidy3", "se_ploidy1", "pe_iupac"])
def test_fastq_bit_exact_vs_instrumented_reference(name, gen, workdir):
    scn = helpers.build_scenario(name, workdir)
    plans, out = helpers.reference_run(scn)
    assert plans
    for i, pf in enumerate(plans):
        plan = planfile.read_plan(pf)
        r1p, r2p = helpers.sample_files(out, plan, i, scn)
        r1, r2 = helpers.read_file(r1p), helpers.read_file(r2p)
        gen.load_plan(plan, scn["seed"])
        f1, f2 = gen.generate()
        assert helpers.first_diff(f1, r1) == -1, "file 1 differs at byte %d" % helpers.first_diff(f1, r1)
        assert helpers.first_diff(f2, r2) == -1, "file 2 differs at byte %d" % helpers.first_diff(f2, r2)
        assert len(r1) > 0


# pass 2 of the fast kernel: a stand-alone move after every batch (what GPUs with fewer than 64 SMs run), or the bulk-copy mover;
# the fast kernel with only the ref == call quality rows in shared memory
OPTION_MODES = {"standalone_move": ("concurrent_move", 0), "concurrent_move": ("concurrent_move", 9), "fast_qmode2": ("fast_qmode", 2)}


@pytest.mark.parametrize("mode", ["force_generic", "fp64_search", "no_splice", "fast_qmode2", "standalone_move", "concurrent_move"])
@pytest.mark.parametrize("name", ["pe_xten", "pe_tiny", "se_gaiix"])
def test_fallback_kernels_bit_exact(name, mode, built, workdir):
    """The generic integer kernel, the FP64 linear-search ground-truth kernel, the fast kernel without the spliced indel path,
    with only the ref == call quality rows in shared memory (the rare substituted bases read the full table in global
    memory), with pass 2 as a stand-alone move after every batch, and with pass 2 on the bulk-copy mover (9 SMs, the default, second
    stream, under the next batch's generation) all give the same bytes, and the statistics name the kernel that ran."""
    from simuscop_b200 import cuda_binding
    scn = helpers.build_scenario(name, workdir)
    plans, out = helpers.reference_run(scn, tag=mode)
    plan = planfile.read_plan(plans[0])
    r1p, r2p = helpers.sample_files(out, plan, 0, scn)
    r1, r2 = helpers.read_file(r1p), helpers.read_file(r2p)
    g = cuda_binding.Generator(0)
    try:
        key, value = OPTION_MODES.get(mode, (mode, 1))
        g.set_option(key, value)
        if key == "concurrent_move":
            g.set_option("batch_pairs", 256)          # many batches: with the mover, every launch but the first moves its predecessor's blobs
        g.load_plan(plan, scn["seed"])
        f1, f2 = g.generate()
        st = g.stats()
    finally:
        g.close()
    assert helpers.first_diff(f1, r1) == -1
    assert helpers.first_diff(f2, r2) == -1
    kernel = {"force_generic": (2, 3), "fp64_search": (4,)}.get(mode, (1,))
    assert st["gen_kernel"] in kernel, st
    if mode == "fast_qmode2":
        rl = plan.hdr["read_length"]
        assert (st["gen_nch"], st["gen_qmode"]) == (2 if rl <= 64 else (rl + 31) // 32, 2), st


def test_error_in_a_pipelined_call_leaves_the_handle_usable(built, workdir):
    """A sink error in the middle of ssc_generate (later batches generated, scanned or moving on the mover's stream) drains
    the device and leaves no batch pending: the same handle's next ssc_generate and ssc_generate_device give the reference's
    bytes and counts."""
    from simuscop_b200 import cuda_binding
    scn = helpers.build_scenario("pe_tiny", workdir)
    plans, out = helpers.reference_run(scn, tag="err")
    plan = planfile.read_plan(plans[0])
    r1p, r2p = helpers.sample_files(out, plan, 0, scn)
    r1, r2 = helpers.read_file(r1p), helpers.read_file(r2p)
    calls = []

    def failing_sink(user, b1, l1, b2, l2, first, n):
        calls.append(n)
        return 1 if len(calls) == 3 else 0
    g = cuda_binding.Generator(0)
    try:
        g.set_option("batch_pairs", 256)
        g.load_plan(plan, scn["seed"])
        assert g.emitted > 4 * 256
        with pytest.raises(cuda_binding.SscError) as e:
            g.generate(sink=failing_sink)
        assert "ssc error 5" in str(e.value) and len(calls) == 3
        f1, f2 = g.generate()
        assert helpers.first_diff(f1, r1) == -1 and helpers.first_diff(f2, r2) == -1
        d = g.generate_device()
        assert (d["bytes1"], d["bytes2"]) == (len(r1), len(r2))
        f1, f2 = g.generate()
        assert helpers.first_diff(f1, r1) == -1 and helpers.first_diff(f2, r2) == -1
    finally:
        g.close()


def test_batching_and_ranges_are_seamless(built, workdir):
    """Small batches and split pair ranges concatenate to the single-shot output (sharding by pair ID)."""
    from simuscop_b200 import cuda_binding
    scn = helpers.build_scenario("pe_tiny", workdir)
    plans, out = helpers.reference_run(scn, tag="rng")
    plan = planfile.read_plan(plans[0])
    g = cuda_binding.Generator(0)
    try:
        g.load_plan(plan, scn["seed"])
        whole1, whole2 = g.generate()
        g.set_option("batch_pairs", 64)
        b1, b2 = g.generate()
        assert (b1, b2) == (whole1, whole2)
        n = g.planned
        cuts = [0, n // 3, n // 3 + 1, 2 * n // 3, n]
        p1 = b"".join(g.generate(a, b)[0] for a, b in zip(cuts[:-1], cuts[1:]))
        p2 = b"".join(g.generate(a, b)[1] for a, b in zip(cuts[:-1], cuts[1:]))
        assert (p1, p2) == (whole1, whole2)
    finally:
        g.close()


@pytest.mark.parametrize("name", ["pe_xten", "pe_variants", "pe_wes", "se_tumor", "pe_tiny", "pe_iupac"])
def test_cli_end_to_end_matches_instrumented_reference(name, built, workdir):
    """The drop-in `simuReads <config>` (C++ front end -> C ABI -> CUDA) writes the same FASTQ files."""
    import glob
    import os
    import subprocess
    from simuscop_b200 import paths, synth
    scn = helpers.build_scenario(name, workdir)
    plans, out_ref = helpers.reference_run(scn, tag="e2e")
    d = scn["dir"]
    out_ours = os.path.join(d, "out_cli")
    cfg = os.path.join(d, "cfg_cli.txt")
    synth.write_config(cfg, output=out_ours, **scn["kw"])
    env = dict(os.environ, SIMUSCOP_SEED=str(scn["seed"]), SIMUSCOP_BATCH_PAIRS="4096")
    r = subprocess.run([paths.SIMUREADS, cfg], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    ref_files = sorted(os.path.basename(f) for f in glob.glob(os.path.join(out_ref, "*.fq")))
    our_files = sorted(os.path.basename(f) for f in glob.glob(os.path.join(out_ours, "*.fq")))
    assert ref_files == our_files and ref_files
    for f in ref_files:
        a, b = helpers.read_file(os.path.join(out_ref, f)), helpers.read_file(os.path.join(out_ours, f))
        assert helpers.first_diff(a, b) == -1, "%s differs at byte %d" % (f, helpers.first_diff(a, b))


def test_cli_sharded_over_two_handles_is_byte_identical(built, workdir):
    """SIMUSCOP_DEVICES shards every sample by pair-ID range (one host thread + one handle per entry); the ordered
    concatenation equals the single-handle output.  "0,0" exercises the path on a single-GPU box."""
    import os
    import subprocess
    import torch
    from simuscop_b200 import paths, synth
    scn = helpers.build_scenario("pe_variants", workdir)
    d = scn["dir"]
    outs = {}
    devs = "0,1,0" if torch.cuda.device_count() >= 2 else "0,0,0"
    for tag, env_extra in (("one", {}), ("three", {"SIMUSCOP_DEVICES": devs})):
        out = os.path.join(d, "out_sh_" + tag)
        cfg = os.path.join(d, "cfg_sh_%s.txt" % tag)
        synth.write_config(cfg, output=out, **scn["kw"])
        env = dict(os.environ, SIMUSCOP_SEED=str(scn["seed"]), SIMUSCOP_BATCH_PAIRS="8192", **env_extra)
        r = subprocess.run([paths.SIMUREADS, cfg], env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        outs[tag] = (helpers.read_file(os.path.join(out, "test_1.fq")), helpers.read_file(os.path.join(out, "test_2.fq")))
        assert sorted(os.listdir(out)) == ["test_1.fq", "test_2.fq"]
    assert outs["one"] == outs["three"] and len(outs["one"][0]) > 0
    # the same sharded run with gzip output: the shard files are concatenated gzip members, a valid .gz of the same bytes
    import gzip
    out = os.path.join(d, "out_sh_gz")
    cfg = os.path.join(d, "cfg_sh_gz.txt")
    synth.write_config(cfg, output=out, **scn["kw"])
    env = dict(os.environ, SIMUSCOP_SEED=str(scn["seed"]), SIMUSCOP_BATCH_PAIRS="8192", SIMUSCOP_DEVICES=devs, SIMUSCOP_GZIP="1")
    r = subprocess.run([paths.SIMUREADS, cfg], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert sorted(os.listdir(out)) == ["test_1.fq.gz", "test_2.fq.gz"]
    assert gzip.decompress(helpers.read_file(os.path.join(out, "test_1.fq.gz"))) == outs["one"][0]
    assert gzip.decompress(helpers.read_file(os.path.join(out, "test_2.fq.gz"))) == outs["one"][1]


@pytest.mark.parametrize("name", sorted(helpers.STRESS))
def test_synthetic_profiles_cli_and_abi(name, built, workdir):
    """Odd k-mer sizes / read lengths / indel rates / degenerate rows: reference == oracle == CUDA (whichever kernel
    variant the configuration selects) == forced generic kernel, through the ABI and through the CLI."""
    import glob
    import os
    import subprocess
    from oracle import binding as oracle_binding
    from simuscop_b200 import cuda_binding, paths, synth
    scn = helpers.build_stress(name, workdir)
    plans, out_ref = helpers.reference_run(scn, tag="st")
    plan = planfile.read_plan(plans[0])
    r1p, r2p = helpers.sample_files(out_ref, plan, 0, scn)
    r1, r2 = helpers.read_file(r1p), helpers.read_file(r2p)
    assert len(r1) > 10000
    o1, o2, _ = oracle_binding.generate(plan, scn["seed"])
    assert (o1, o2) == (r1, r2)
    for opt in (None, "force_generic", "no_splice"):
        g = cuda_binding.Generator(0)
        try:
            if opt:
                g.set_option(opt, 1)
            g.load_plan(plan, scn["seed"])
            f1, f2 = g.generate()
        finally:
            g.close()
        assert helpers.first_diff(f1, r1) == -1, (opt, helpers.first_diff(f1, r1))
        assert helpers.first_diff(f2, r2) == -1, (opt, helpers.first_diff(f2, r2))
    d = scn["dir"]
    cfg = os.path.join(d, "cfg_cli.txt")
    synth.write_config(cfg, output=os.path.join(d, "out_cli"), **scn["kw"])
    r = subprocess.run([paths.SIMUREADS, cfg], env=dict(os.environ, SIMUSCOP_SEED=str(scn["seed"])), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    for f in glob.glob(os.path.join(out_ref, "*.fq")):
        assert helpers.read_file(f) == helpers.read_file(os.path.join(d, "out_cli", os.path.basename(f)))


def test_reads_beyond_the_scratch_limits_fail_loudly(built, workdir):
    """A profile with 2 % insertion AND deletion rates outgrows the per-read limits (32 events / 128 inserted bases):
    the library must return SSC_ERR_OVERFLOW, not a silently different FASTQ, from both pipelined calls.  The handle stays
    usable: the next plan loaded on it gives the reference's bytes."""
    from simuscop_b200 import cuda_binding
    scn = helpers.build_stress("overflow", workdir)
    plans, out_ref = helpers.reference_run(scn, tag="ov")
    plan = planfile.read_plan(plans[0])
    tiny = helpers.build_scenario("pe_tiny", workdir)
    tiny_plans, tiny_out = helpers.reference_run(tiny, tag="ov")
    tiny_plan = planfile.read_plan(tiny_plans[0])
    t1, t2 = (helpers.read_file(p) for p in helpers.sample_files(tiny_out, tiny_plan, 0, tiny))
    for opt in (None, "force_generic", "no_splice"):
        g = cuda_binding.Generator(0)
        try:
            if opt:
                g.set_option(opt, 1)
            g.load_plan(plan, scn["seed"])
            with pytest.raises(cuda_binding.SscError) as e:
                g.generate()
            assert "ssc error 6" in str(e.value)
            with pytest.raises(cuda_binding.SscError) as e:
                g.generate_device()
            assert "ssc error 6" in str(e.value)
            g.load_plan(tiny_plan, tiny["seed"])
            f1, f2 = g.generate()
            assert helpers.first_diff(f1, t1) == -1 and helpers.first_diff(f2, t2) == -1
        finally:
            g.close()


def test_gc_census_matches_host_counts(built, workdir):
    """ssc_gc_census (device half of Segment::getWeightedLength / calculateGCPercent) against numpy on the same
    haplotype string: random, empty, single-base, word-straddling and whole-store intervals, N runs, lower case,
    and a profile whose base order puts G on code 0 (the code non-ACGT bases are stored with)."""
    import numpy as np
    from simuscop_b200 import cuda_binding
    rng = np.random.default_rng(11)
    for stress in ("k3_rl95", "k3_fixed_insert_pe"):            # base orders ACTG and GATC
        scn = helpers.build_stress(stress, workdir)
        plans, _ = helpers.reference_run(scn, tag="gc")
        plan = planfile.read_plan(plans[0])
        g = cuda_binding.Generator(0)
        try:
            g.load_plan(plan, scn["seed"])
            hap = np.frombuffer(bytes(plan.genome), np.uint8)
            n = len(hap)
            up = hap & 0xDF                                      # upper case
            is_gc = (up == ord("G")) | (up == ord("C"))
            is_n = ~((up == ord("A")) | (up == ord("C")) | (up == ord("G")) | (up == ord("T")))
            assert is_n.any()
            cg = np.concatenate(([0], np.cumsum(is_gc & ~is_n)))
            cn = np.concatenate(([0], np.cumsum(is_n)))
            starts = rng.integers(0, n, 4000)
            lens = np.minimum(rng.integers(0, 3000, 4000), n - starts)
            starts = np.concatenate((starts, [0, 0, n - 1, n, 5, 31, 32, 33, 0]))
            lens = np.concatenate((lens, [0, 1, 1, 0, 27, 1, 1, 64, n]))
            # 1 kb windows exactly as the plan uses them
            starts = np.concatenate((starts, np.arange(0, n - 1000, 1000)))
            lens = np.concatenate((lens, np.full(len(np.arange(0, n - 1000, 1000)), 1000)))
            gc, nn = g.gc_census(starts, lens)
            assert (gc == cg[starts + lens] - cg[starts]).all()
            assert (nn == cn[starts + lens] - cn[starts]).all()
            with pytest.raises(cuda_binding.SscError):
                g.gc_census([n - 3], [10])                       # interval past the store
        finally:
            g.close()


def test_device_plan_equals_host_plan(built, workdir):
    """The plan built with the GPU weights pass (haplotype upload + ssc_gc_census) is the plan of the host-only pass:
    the CLI's plan dump with a device is byte-identical to the SIMUSCOP_PLAN_ONLY dump (which test_host_logic pins
    against the instrumented reference), for WGS with variants, WES targets and a tumour mixture."""
    import os
    import subprocess
    from simuscop_b200 import paths, synth
    for name in ("pe_variants", "pe_wes", "se_tumor", "pe_iupac"):
        scn = helpers.build_scenario(name, workdir)
        d = scn["dir"]
        dumps = {}
        for tag, extra in (("host", {"SIMUSCOP_PLAN_ONLY": "1"}), ("dev", {})):
            cfg = os.path.join(d, "cfg_plan_%s.txt" % tag)
            synth.write_config(cfg, output=os.path.join(d, "out_plan_" + tag), **scn["kw"])
            prefix = os.path.join(d, "plan_%s" % tag)
            env = dict(os.environ, SIMUSCOP_SEED=str(scn["seed"]), SIMUSCOP_DUMP_PLAN=prefix, **extra)
            r = subprocess.run([paths.SIMUREADS, cfg], env=env, capture_output=True, text=True)
            assert r.returncode == 0, r.stderr[-2000:]
            files = sorted(f for f in os.listdir(d) if f.startswith("plan_%s" % tag))
            assert files
            dumps[tag] = [helpers.read_file(os.path.join(d, f)) for f in files]
        assert len(dumps["host"]) == len(dumps["dev"])
        for a, b in zip(dumps["host"], dumps["dev"]):
            assert a == b


@pytest.mark.parametrize("name,batch", [("pe_xten", 0), ("pe_xten", 4096), ("se_ploidy1", 0), ("pe_tiny", 0)])
def test_gzip_output_inflates_to_the_plain_fastq(name, batch, built, workdir):
    """ssc_set_option("gzip", 1): the slabs are concatenated gzip members compressed on the GPU (one per 32-record
    blob, literal-only dynamic Huffman blocks, CRC-32 + ISIZE trailers checked by zlib); inflated they are byte for
    byte the plain output, which is the instrumented reference's."""
    import gzip
    from simuscop_b200 import cuda_binding
    scn = helpers.build_scenario(name, workdir)
    plans, out = helpers.reference_run(scn, tag="gz")
    plan = planfile.read_plan(plans[0])
    r1p, r2p = helpers.sample_files(out, plan, 0, scn)
    r1, r2 = helpers.read_file(r1p), helpers.read_file(r2p)
    g = cuda_binding.Generator(0)
    try:
        g.set_option("gzip", 1)
        if batch:
            g.set_option("batch_pairs", batch)
        g.load_plan(plan, scn["seed"])
        z1, z2 = g.generate()
        st = g.stats()
        assert gzip.decompress(z1) == r1
        assert (gzip.decompress(z2) if z2 else b"") == r2
        assert st["fastq_bytes"] == len(r1) + len(r2) and st["gz_bytes"] == len(z1) + len(z2)
        assert len(z1) < 0.6 * len(r1)          # ~0.3 with XTen's 7 quality symbols, ~0.5 with 40
        # back to plain output on the same handle
        g.set_option("gzip", 0)
        f1, f2 = g.generate()
        assert f1 == r1 and f2 == r2
    finally:
        g.close()


def test_cli_gzip_files(built, workdir):
    """SIMUSCOP_GZIP=1: <name>_1.fq.gz / _2.fq.gz inflate to the files of the plain run."""
    import gzip
    import os
    import subprocess
    from simuscop_b200 import paths, synth
    scn = helpers.build_scenario("pe_xten", workdir)
    d = scn["dir"]
    outs = {}
    for tag, env in (("plain", {}), ("gz", {"SIMUSCOP_GZIP": "1"})):
        out = os.path.join(d, "out_clig_" + tag)
        cfg = os.path.join(d, "cfg_clig_%s.txt" % tag)
        synth.write_config(cfg, output=out, **scn["kw"])
        r = subprocess.run([paths.SIMUREADS, cfg], env=dict(os.environ, SIMUSCOP_SEED=str(scn["seed"]), **env), capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
        outs[tag] = out
    assert sorted(os.listdir(outs["gz"])) == ["test_1.fq.gz", "test_2.fq.gz"]
    for k in ("1", "2"):
        assert gzip.decompress(helpers.read_file(os.path.join(outs["gz"], "test_%s.fq.gz" % k))) == \
            helpers.read_file(os.path.join(outs["plain"], "test_%s.fq" % k))


@pytest.mark.parametrize("ctas", [1, 3])
def test_many_tickets_per_warp(ctas, built, workdir):
    """At full size a warp of the generation kernel works through a dozen tickets of 32 pairs one after the other; the
    parity scenarios are small enough for one ticket per warp.  Capping the grid makes every warp take many tickets
    (shared-memory windows, headers and indel scratch are reused across pairs and tickets) -- same bytes, plain and gzip."""
    import gzip
    from simuscop_b200 import cuda_binding
    for name in ("pe_xten", "pe_variants"):
        scn = helpers.build_scenario(name, workdir)
        plans, out = helpers.reference_run(scn, tag="mt")
        plan = planfile.read_plan(plans[0])
        r1p, r2p = helpers.sample_files(out, plan, 0, scn)
        r1, r2 = helpers.read_file(r1p), helpers.read_file(r2p)
        g = cuda_binding.Generator(0)
        try:
            g.set_option("max_ctas", ctas)
            g.load_plan(plan, scn["seed"])
            f1, f2 = g.generate()
            assert helpers.first_diff(f1, r1) == -1 and helpers.first_diff(f2, r2) == -1
            g.set_option("gzip", 1)
            z1, z2 = g.generate()
            assert gzip.decompress(z1) == r1 and gzip.decompress(z2) == r2
        finally:
            g.close()


@pytest.mark.parametrize("name", ["pe_variants", "se_tumor", "pe_ploidy3", "pe_xten"])
def test_device_built_haplotypes_equal_host_strings(name, built, workdir):
    """SURVEY 8f rank 2: segments without indel variants are built on the device from the uploaded chromosome
    (ssc_reference_upload / ssc_genome_append_ref / ssc_genome_poke: copies per copy-number phasing + SNP / SNV alleles);
    the decoded store must equal the haplotype strings the host builds (the plan dump, pinned against the instrumented
    reference by test_host_logic), base for base, for every sample."""
    import os
    import numpy as np
    from simuscop_b200 import cuda_binding, host_binding, synth
    scn = helpers.build_scenario(name, workdir)
    d = scn["dir"]
    cfg = os.path.join(d, "cfg_hap.txt")
    synth.write_config(cfg, output=os.path.join(d, "out_hap"), **scn["kw"])
    job = host_binding.Job(cfg, scn["seed"])
    g = cuda_binding.Generator(0)
    try:
        for s in range(job.num_samples):
            dump = os.path.join(d, "hap_%d.plan" % s)
            job.prepare(s, g, dump)
            plan = planfile.read_plan(dump)
            want = np.frombuffer(bytes(plan.genome), np.uint8).copy()
            want &= 0xDF                                                      # upper case
            ok = (want == ord("A")) | (want == ord("C")) | (want == ord("G")) | (want == ord("T"))
            want[~ok] = ord("N")
            assert g.genome_size() == len(want)
            got = np.frombuffer(g.genome_read(0, len(want)), np.uint8)
            assert (got == want).all(), "first difference at store base %d" % int(np.flatnonzero(got != want)[0])
    finally:
        g.close()
        job.close()


def test_fasta_record_unfolded_on_the_device(built, tmp_path):
    """ssc_reference_upload_fasta: the sequence lines of a FASTA record read from the file descriptor and unfolded on the GPU
    (line ends dropped, upper-cased) equal the host's chromosome string, for several line geometries (60 / 7 / 1000 columns,
    CR-LF line ends, a last line with and without terminator, a record in the middle of the file), and the count of characters
    that are neither ACGT nor N is exact."""
    import ctypes as C
    import os
    import numpy as np
    from simuscop_b200 import cuda_binding
    rng = np.random.default_rng(17)
    L = cuda_binding.lib()
    scn = helpers.build_stress("k3_rl95", str(tmp_path))
    plans, _ = helpers.reference_run(scn, tag="uf")
    plan = planfile.read_plan(plans[0])
    g = cuda_binding.Generator(0)
    try:
        g.load_plan(plan, scn["seed"])                       # a profile must be set (base order of the packed codes)
        for cols, eol, n, tail_eol in ((60, b"\n", 100000, True), (7, b"\n", 1234, False), (1000, b"\r\n", 2501, True),
                                       (60, b"\n", 60, True), (61, b"\n", 1, False), (50, b"\n", 3000017, True)):
            seq = np.frombuffer(b"ACGTacgtNnRYkm", np.uint8)[rng.integers(0, 14, n)]
            body = b"".join(seq[i:i + cols].tobytes() + eol for i in range(0, n, cols))
            if not tail_eol:
                body = body[:-len(eol)]
            head = b">first\nACGT\n>chrT some text\n"
            path = str(tmp_path / ("g_%d_%d.fa" % (cols, n)))
            with open(path, "wb") as f:
                f.write(head + body + (b"\n>after\nGGGG\n" if tail_eol else b""))
            lines = (n - 1) // cols
            raw_len = n + lines * len(eol)
            fd = os.open(path, os.O_RDONLY)
            other = C.c_uint64()
            try:
                cuda_binding._ck(L.ssc_reference_upload_fasta(g.h, fd, len(head), raw_len, n, cols, cols + len(eol), C.byref(other)))
            finally:
                os.close(fd)
            up = seq & 0xDF
            is_acgtn = (up == 65) | (up == 67) | (up == 71) | (up == 84) | (up == 78)
            assert other.value == int((~is_acgtn).sum())
            cuda_binding._ck(L.ssc_genome_reserve(g.h, 2 * n + 64))
            first = C.c_uint64()
            cuda_binding._ck(L.ssc_genome_append_ref(g.h, 0, n, 2, C.byref(first)))
            want = up.copy()
            want[~((up == 65) | (up == 67) | (up == 71) | (up == 84))] = ord("N")
            got = np.frombuffer(g.genome_read(0, 2 * n), np.uint8)
            assert (got[:n] == want).all() and (got[n:] == want).all(), (cols, n)
    finally:
        g.close()
