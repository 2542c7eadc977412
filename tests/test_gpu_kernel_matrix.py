"""Every instance of the generation kernel against the C oracle (oracle/ssc_oracle.c, the FP64 linear-search restatement that
test_oracle_pinning pins against the instrumented reference), byte for byte, at the read lengths, table shapes and
shared-memory budgets where the instances differ.

The fast kernel is compiled as generate_slots_kernel<NCH, QP>: NCH = 2..5 chunks of 32 cycles (from the read length), QP = where
the quality tables live (8: every row in shared memory as 32-bit thresholds, 16: every row as 16-bit keys with an exact repeat
on ties, 2: only the ref == call rows, 0: everything in global memory; chosen from the profile and the shared-memory budget).
The generic kernels take what the fast one cannot: K != 3, RL 161..320, tables too large.  Every case asserts the instance
that ran (ssc_stats gen_kernel / gen_nch / gen_qmode), so that a change of the selection or of the shared-memory footprint
cannot move a case off the instance it names without failing.  The expected instances follow from the B200's shared-memory
budget (sharedMemPerBlockOptin 232 448 bytes); on another device only the bytes are compared.

The plans come from the C++ front end in plan-only mode on synthetic profiles (simuscop_b200.synth.write_profile) and genomes
with N runs, lower case and IUPAC codes; each plan is generated once by the oracle."""
import os
import subprocess

import pytest

import helpers
from simuscop_b200 import planfile, synth, testdata

pytestmark = pytest.mark.gpu

B200_SMEM_OPTIN = 232448
FAST, GENERIC_SMEM, GENERIC_GLOBAL, FP64 = 1, 2, 3, 4


def fast_nch(rl):
    return 2 if rl <= 64 else (rl + 31) // 32


def _synthetic(rl, bins, live, layout="PE", bases="ACTG", kmer=3, rates=(3e-3, 3e-3), std_isize=30.0, lengths=(60000, 9000),
               coverage=8):
    return dict(profile_kw=dict(kmer=kmer, read_length=rl, bins=bins, n_live_qual=live, bases=bases, ins_rate=rates[0],
                                del_rate=rates[1], std_isize=std_isize),
                layout=layout, insertSize=rl + 90, lengths=lengths, coverage=coverage)


def _shipped(profile, rl, layout="PE", lengths=(60000, 9000), coverage=4):
    return dict(profile=profile, layout=layout, insertSize=rl + 150, lengths=lengths, coverage=coverage)


# a. read-length edges: K = 3 and 5..8 live quality symbols (quality rows of 8 entries), so that every quality mode can be
# forced and fits (B <= 50); the record tail of the fast kernel depends on RL % 32, and RL = 32 * NCH sends every read with
# a net insertion past the unrolled chunks.  Bins: 1, odd, B == RL; PE and SE; base orders; one fixed-insert PE profile
# (use_cdf2 = 0: mate 2 reads substitution table 1).  About 0.55 Mbases each.
EDGE = {
    33: _synthetic(33, 33, 7, "SE"),
    62: _synthetic(62, 1, 5, "PE", "GATC", rates=(2.5e-3, 3.5e-3)),
    63: _synthetic(63, 21, 6, "SE", "TCGA"),
    64: _synthetic(64, 31, 7, "PE", "CATG", std_isize=0.0),
    65: _synthetic(65, 13, 8, "PE", "ACGT"),
    94: _synthetic(94, 47, 6, "SE", "GTAC", rates=(3.5e-3, 2.5e-3)),
    95: _synthetic(95, 45, 7, "PE"),
    96: _synthetic(96, 1, 5, "PE", "TGCA"),
    97: _synthetic(97, 49, 8, "SE"),
    126: _synthetic(126, 25, 7, "PE", "AGCT"),
    127: _synthetic(127, 39, 6, "PE", "CTAG", rates=(3.5e-3, 3e-3)),
    128: _synthetic(128, 43, 7, "PE"),
    129: _synthetic(129, 1, 5, "SE", "GCTA"),
    158: _synthetic(158, 35, 7, "PE", "TACG"),
    159: _synthetic(159, 49, 6, "SE"),
    160: _synthetic(160, 41, 7, "PE", "CATG", rates=(3e-3, 3.5e-3)),
}
QMODES = (8, 16, 2, 0)

# b. full-width quality rows: exactly 40 live symbols (every key of a 16-bit row is live; natural QP 16), one NCH each, at
# 3.5 Mbases (about 9 sixteen-bit compares per base, each a tie with probability 2^-16: some 500 exact repeats per run);
# 41 live symbols (past the 16-bit rows: natural QP 2); 4 live symbols at RL 151 (binned qualities: rows of 4 rule out QP 8)
BIG = dict(lengths=(300000, 90000), coverage=9)
WIDE = {
    "q40_rl64": (_synthetic(64, 31, 40, "PE", **BIG), (FAST, 2, 16)),
    "q40_rl96": (_synthetic(96, 45, 40, "SE", "GATC", **BIG), (FAST, 3, 16)),
    "q40_rl128": (_synthetic(128, 37, 40, "PE", "TGCA", **BIG), (FAST, 4, 16)),
    "q40_rl160": (_synthetic(160, 49, 40, "PE", **BIG), (FAST, 5, 16)),
    "q41_rl100": (_synthetic(100, 41, 41, "PE", coverage=15), (FAST, 4, 2)),
    "q4_rl151": (_synthetic(151, 50, 4, "PE", **BIG), (FAST, 5, 16)),
}

# c. what the selection picks at the edges of the shared-memory budget: XTen (the benchmark's profile; QP 8 takes 226 352 of
# the 231 424 bytes here), the 40-symbol shipped profiles, K = 3 PE profiles with 20 live symbols as the bins grow (QP 16 -> 2 -> 0 -> the
# generic kernel), SE with 100 bins and 40 symbols, and the read lengths just outside the fast kernel
BUDGET = {
    "xten_rl151": (_shipped("XTen", 150), (FAST, 5, 8)),
    "hiseq2500": (_shipped("HiSeq2500", 125), (FAST, 4, 16)),
    "gaiix": (_shipped("GAIIx", 100, "SE"), (FAST, 3, 16)),
    "pe_b56": (_synthetic(120, 56, 20, "PE"), (FAST, 4, 16)),
    "pe_b62": (_synthetic(90, 62, 20, "PE", "GATC"), (FAST, 3, 2)),
    "pe_b70": (_synthetic(150, 70, 20, "PE"), (FAST, 5, 0)),
    "pe_b76": (_synthetic(100, 76, 20, "PE"), (GENERIC_GLOBAL, 10, -1)),
    "se_b100_q40": (_synthetic(140, 100, 40, "SE"), (FAST, 5, 0)),
    "rl32": (_synthetic(32, 15, 7, "PE"), (GENERIC_SMEM, 10, -1)),
    "rl161": (_synthetic(161, 23, 7, "PE"), (GENERIC_SMEM, 10, -1)),
}

# d. the generic kernels: long reads with the K = 3 tables in shared memory and, with 76 bins or more, in global memory;
# K = 5 and K = 8 (the documented limit); the FP64 linear search
GENERIC = {
    "rl161_b20": (_synthetic(161, 20, 7, "PE", coverage=4), (GENERIC_SMEM, 10, -1)),
    "rl256_b31": (_synthetic(256, 31, 12, "PE", "GATC", coverage=4), (GENERIC_SMEM, 10, -1)),
    "rl320_b45": (_synthetic(320, 45, 7, "SE", coverage=4), (GENERIC_SMEM, 10, -1)),
    "rl161_b80": (_synthetic(161, 80, 7, "PE", coverage=4), (GENERIC_GLOBAL, 10, -1)),
    "rl256_b91": (_synthetic(256, 91, 20, "PE", "TCGA", coverage=4), (GENERIC_GLOBAL, 10, -1)),
    "rl320_b76": (_synthetic(320, 76, 7, "PE", coverage=4), (GENERIC_GLOBAL, 10, -1)),
    "k5_b3": (_synthetic(100, 3, 7, "PE", kmer=5), (GENERIC_GLOBAL, 10, -1)),
    "k8_b2": (_synthetic(90, 2, 6, "PE", "GATC", kmer=8, coverage=4), (GENERIC_GLOBAL, 10, -1)),
}

CASES = {"rl%d" % rl: spec for rl, spec in EDGE.items()}
for table in (WIDE, BUDGET, GENERIC):
    CASES.update({name: spec for name, (spec, _) in table.items()})
CASES["rl321"] = _synthetic(321, 40, 7, "PE", coverage=1)      # one past the longest supported read


def build_case(name, workdir):
    """Genome, profile and config of CASES[name] under `workdir`; the scenario dict of tests/helpers.py."""
    spec = CASES[name]
    d = os.path.join(workdir, "km_" + name)
    os.makedirs(d, exist_ok=True)
    ref = os.path.join(d, "ref.fa")
    synth.make_genome(ref, list(spec["lengths"]), seed=31, n_runs=2, lower_runs=2, run_len=200, iupac=40)
    if "profile" in spec:
        data = testdata.materialize(os.path.join(workdir, "data"))
        prof = os.path.join(data, testdata.PROFILES[spec["profile"]])
    else:
        prof = os.path.join(d, "synthetic.profile")
        synth.write_profile(prof, seed=sum(map(ord, name)), **spec["profile_kw"])
    kw = dict(ref=ref, profile=prof, layout=spec["layout"], coverage=spec["coverage"], insertSize=spec["insertSize"], threads=1,
              verbose=0, name="km")
    return dict(dir=d, kw=kw, seed=5, name=name)


@pytest.fixture(scope="module")
def reference(built, workdir):
    """name -> (plan, seed, oracle FASTQ 1, oracle FASTQ 2), each plan built and generated once."""
    from oracle import binding as oracle_binding
    cache = {}

    def get(name):
        if name not in cache:
            scn = build_case(name, workdir)
            plan = planfile.read_plan(helpers.plan_dumps(scn, "km")[0])
            f1, f2, info = oracle_binding.generate(plan, scn["seed"])
            assert info["bases"] > 100000
            cache[name] = (plan, scn["seed"], f1, f2)
        return cache[name]
    return get


@pytest.fixture(scope="module")
def check_path(built):
    """Asserts the instance a run launched, (gen_kernel, gen_nch, gen_qmode), where the expectation holds: on a device with the
    B200's shared-memory budget."""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin

    def check(stats, want):
        if optin == B200_SMEM_OPTIN:
            assert (stats["gen_kernel"], stats["gen_nch"], stats["gen_qmode"]) == want, stats
    return check


def run_gpu(plan, seed, **options):
    """One handle, the given ssc_set_option keys (before the profile), the whole plan; returns (FASTQ 1, FASTQ 2, stats)."""
    from simuscop_b200 import cuda_binding
    g = cuda_binding.Generator(0)
    try:
        for k, v in options.items():
            g.set_option(k, v)
        g.load_plan(plan, seed)
        f1, f2 = g.generate()
        return f1, f2, g.stats()
    finally:
        g.close()


def _record(data, rec):
    lines = data.split(b"\n")[4 * rec:4 * rec + 4]
    return b"\n".join(lines)


def assert_same_fastq(got, want, what):
    for f, (a, b) in enumerate(zip(got, want)):
        i = helpers.first_diff(a, b)
        if i != -1:
            rec = b.count(b"\n", 0, i) // 4
            pytest.fail("%s: file %d differs from the oracle at byte %d, record %d (%d vs %d bytes)\n  oracle: %r\n  gpu:    %r"
                        % (what, f + 1, i, rec, len(b), len(a), _record(b, rec), _record(a, rec)))


def _edge_params():
    out = []
    for rl in EDGE:
        for q in QMODES:
            for splice in (True, False):
                out.append(pytest.param(rl, q, splice, id="rl%d-nch%d-qp%d%s" % (rl, fast_nch(rl), q, "" if splice else "-nosplice")))
        out.append(pytest.param(rl, None, True, id="rl%d-generic-smem" % rl))
    return out


@pytest.mark.parametrize("rl,qmode,splice", _edge_params())
def test_read_length_edges(rl, qmode, splice, reference, check_path):
    """Every (NCH, QP) instance, forced with fast_qmode, with and without the spliced indel path, and the generic kernel
    (force_generic), at read lengths on both sides of every 32-cycle chunk boundary: the same bytes as the oracle."""
    plan, seed, o1, o2 = reference("rl%d" % rl)
    options = {"force_generic": 1} if qmode is None else {"fast_qmode": qmode, "no_splice": 0 if splice else 1}
    f1, f2, st = run_gpu(plan, seed, **options)
    assert_same_fastq((f1, f2), (o1, o2), "RL %d, %s" % (rl, options))
    check_path(st, (GENERIC_SMEM, 10, -1) if qmode is None else (FAST, fast_nch(rl), qmode))


def _ids(table):
    return [pytest.param(name, want, id="%s-%s" % (name, "nch%d-qp%d" % want[1:] if want[0] == FAST else
                                                  {GENERIC_SMEM: "generic-smem", GENERIC_GLOBAL: "generic-global"}[want[0]]))
            for name, (_, want) in table.items()]


@pytest.mark.parametrize("name,want", _ids(WIDE))
def test_full_width_quality_rows(name, want, reference, check_path):
    """Quality rows with exactly 40 live symbols run the 16-bit-key tables with every key live, long enough that hundreds of
    draws tie with a key and repeat the lookup on the exact tables; 41 symbols fall back to the ref == call rows; 4 symbols
    (binned qualities) run the 16-bit tables at RL 151."""
    plan, seed, o1, o2 = reference(name)
    f1, f2, st = run_gpu(plan, seed)
    assert_same_fastq((f1, f2), (o1, o2), name)
    check_path(st, want)


@pytest.mark.parametrize("name,qmode", [pytest.param("q4_rl151", 8, id="q4_rl151-qp8-generic-smem"),
                                        pytest.param("q41_rl100", 16, id="q41_rl100-qp16-generic-smem")])
def test_forced_mode_that_does_not_apply(name, qmode, reference, check_path):
    """A quality mode forced on a profile that cannot use it (QP 8 needs rows of 5..8 live symbols, QP 16 at most 40) leaves
    the profile to the generic kernel, which gives the same bytes."""
    plan, seed, o1, o2 = reference(name)
    f1, f2, st = run_gpu(plan, seed, fast_qmode=qmode)
    assert_same_fastq((f1, f2), (o1, o2), "%s, fast_qmode %d" % (name, qmode))
    check_path(st, (GENERIC_SMEM, 10, -1))


@pytest.mark.parametrize("name,want", _ids(BUDGET))
def test_selection_at_the_budget_edges(name, want, reference, check_path):
    """What the automatic selection runs when the tables approach the shared-memory budget, and just outside the read lengths
    of the fast kernel: the same bytes as the oracle, on the instance named in the test id."""
    plan, seed, o1, o2 = reference(name)
    f1, f2, st = run_gpu(plan, seed)
    assert_same_fastq((f1, f2), (o1, o2), name)
    check_path(st, want)


@pytest.mark.parametrize("name,want", _ids(GENERIC))
def test_generic_kernel_edges(name, want, reference, check_path):
    """The generic kernel at RL 161, 256 and 320 with its K = 3 tables in shared memory and, under force_generic with 76 bins
    or more, in global memory; K = 5 and K = 8."""
    plan, seed, o1, o2 = reference(name)
    f1, f2, st = run_gpu(plan, seed, force_generic=1)
    assert_same_fastq((f1, f2), (o1, o2), name)
    check_path(st, want)


@pytest.mark.parametrize("name", ["rl33", "rl160", "rl320_b45"])
def test_fp64_search(name, reference, check_path):
    """The FP64 linear-search kernel at the shortest, the longest fast-kernel and the longest supported read."""
    plan, seed, o1, o2 = reference(name)
    f1, f2, st = run_gpu(plan, seed, fp64_search=1)
    assert_same_fastq((f1, f2), (o1, o2), name)
    check_path(st, (FP64, 10, -1))


def test_read_length_321_is_rejected(built, workdir):
    """Reads longer than 320 are refused, by ssc_set_profile with SSC_ERR_INVALID and by the CLI with a non-zero exit, not
    generated wrongly."""
    from simuscop_b200 import cuda_binding, paths
    scn = build_case("rl321", workdir)
    plan = planfile.read_plan(helpers.plan_dumps(scn, "km")[0])
    with pytest.raises(cuda_binding.SscError) as e:
        run_gpu(plan, scn["seed"])
    assert "ssc error 1" in str(e.value) and "320" in str(e.value)
    cfg = os.path.join(scn["dir"], "cfg_cli.txt")
    synth.write_config(cfg, output=os.path.join(scn["dir"], "out_cli"), **scn["kw"])
    r = subprocess.run([paths.SIMUREADS, cfg], env=dict(os.environ, SIMUSCOP_SEED=str(scn["seed"])), capture_output=True, text=True)
    assert r.returncode != 0, r.stderr[-2000:]


def test_fast_qmode_option(reference):
    """fast_qmode takes -1, 8, 16, 2 and 0, only before ssc_set_profile; the option it replaced is gone; ssc_reset_stats
    clears the instance of the last launch."""
    from simuscop_b200 import cuda_binding
    plan, seed, _, _ = reference("rl33")
    g = cuda_binding.Generator(0)
    try:
        for v in (-1, 8, 16, 2, 0):
            g.set_option("fast_qmode", v)
        for v in (1, 4, 32, -2):
            with pytest.raises(cuda_binding.SscError, match="ssc error 1"):
                g.set_option("fast_qmode", v)
        with pytest.raises(cuda_binding.SscError, match="unknown option"):
            g.set_option("no_q16", 1)
        g.load_plan(plan, seed)
        with pytest.raises(cuda_binding.SscError, match="ssc error 3"):
            g.set_option("fast_qmode", 2)
        g.generate_device()
        assert g.stats()["gen_kernel"] == FAST
        g.reset_stats()
        st = g.stats()
        assert (st["gen_kernel"], st["gen_nch"], st["gen_qmode"], st["gen_smem_bytes"]) == (0, 0, 0, 0)
    finally:
        g.close()
