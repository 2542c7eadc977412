"""Array output (ssc_generate_reads / Generator.generate_reads): the reads of a pair range in caller-owned device arrays.

Every check re-formats the arrays into FASTQ records (segment_name + pos + '#' + frag + '/mate', bases, '+', qualities) and
compares them byte for byte with ssc_generate on the same handle and range, which the parity suites pin to the reference:
on the parity scenarios, on every (NCH, QP) instance of the fast kernel at the read-length edges, with no_splice, many
batches and one CTA, and on the hand-built plans of test_gpu_plan_edges (one-pair bins, 64-byte names, 10-digit fields,
pair IDs past 2^32).  Every output buffer is pre-filled with 0xFF, so that a byte past a read's length the kernel failed to
clear shows up, and the statistics of the two calls agree."""
import ctypes as C
import os

import numpy as np
import pytest

import helpers
from simuscop_b200 import abi, planfile, synth
from test_gpu_kernel_matrix import B200_SMEM_OPTIN, EDGE, FAST, QMODES, fast_nch
from test_gpu_plan_edges import SEED, Builder, cases, dense_case, huge_bins, load, oracle, profiles  # noqa: F401 (fixtures)

pytestmark = pytest.mark.gpu


def prefilled(g, n):
    """Output arrays for n pairs with every byte 0xFF."""
    out = g.empty_reads(n)
    for k in ("reads", "length", "pair_id", "segment", "pos", "frag"):
        out[k].fill_(-1 if out[k].dtype.is_signed else 0xFF)
    return out


def to_fastq(g, a):
    """The FASTQ files the arrays stand for; also asserts that every byte past a read's length is 0."""
    reads = a["reads"].cpu().numpy()
    length = a["length"].cpu().numpy().astype(np.int64)
    seg, pos, frag = (a[k].cpu().numpy() for k in ("segment", "pos", "frag"))
    n, mates, _, pitch = reads.shape
    past = np.arange(pitch)[None, None, None, :] >= length[:, :, None, None]
    assert (reads[np.broadcast_to(past, reads.shape)] == 0).all(), "a byte past a read's length is not 0"
    assert ((length > 0) & (length <= pitch)).all()
    names = {int(s): g.segment_name(int(s)) for s in np.unique(seg)}
    files = [[] for _ in range(mates)]
    for i in range(n):
        head = names[int(seg[i])] + b"%d#%d" % (pos[i], frag[i])
        for m in range(mates):
            ln = length[i, m]
            files[m].append(head + (b"/%d\n" % (m + 1) if mates == 2 else b"\n") + reads[i, m, 0, :ln].tobytes() + b"\n+\n" +
                            reads[i, m, 1, :ln].tobytes() + b"\n")
    return b"".join(files[0]), b"".join(files[1]) if mates == 2 else b""


COUNTS = ("pairs_emitted", "reads_emitted", "bases_emitted")


def check_range(g, lo=0, hi=None, stream=None):
    """Arrays of [lo, hi) == ssc_generate of [lo, hi) on the same handle, with the same pair / read / base counts; returns the arrays."""
    if hi is None:
        hi = g.planned
    g.reset_stats()
    f1, f2 = g.generate(lo, hi)
    want = g.stats()
    n = g.read_shape(lo, hi)[0]
    g.reset_stats()
    a = g.generate_reads(lo, hi, stream=stream, out=prefilled(g, n))
    got = g.stats()
    assert a["reads"].shape[0] == n == got["pairs_emitted"]
    a1, a2 = to_fastq(g, a)
    assert helpers.first_diff(a1, f1) == -1, "file 1 differs at byte %d" % helpers.first_diff(a1, f1)
    assert helpers.first_diff(a2, f2) == -1, "file 2 differs at byte %d" % helpers.first_diff(a2, f2)
    assert [got[k] for k in COUNTS] == [want[k] for k in COUNTS]
    assert got["fastq_bytes"] == 0 and got["gen_kernel"] == FAST
    return a


@pytest.fixture(scope="module")
def gen(built):
    from simuscop_b200 import cuda_binding
    g = cuda_binding.Generator(0)
    yield g
    g.close()


def scenario_plan(name, workdir, tag="arr"):
    scn = helpers.build_scenario(name, workdir)
    return planfile.read_plan(helpers.plan_dumps(scn, tag)[0]), scn["seed"]


@pytest.mark.parametrize("name", ["pe_xten", "se_gaiix", "pe_tiny", "pe_variants", "pe_wes", "se_tumor", "pe_ploidy3", "se_ploidy1",
                                  "pe_iupac"])
def test_parity_scenarios(name, gen, workdir):
    """PE and SE, variants and indels, WES, tumour mixtures, ploidy 1 and 3, IUPAC codes and N runs."""
    plan, seed = scenario_plan(name, workdir)
    gen.load_plan(plan, seed)
    check_range(gen)


@pytest.mark.parametrize("option", [("no_splice", 1), ("batch_pairs", 256), ("max_ctas", 1)])
def test_options(option, built, workdir):
    """Reads with indel events on the position-by-position path; many batches, each written at its row offset; one CTA, whose
    warps take many tickets."""
    from simuscop_b200 import cuda_binding
    plan, seed = scenario_plan("pe_variants", workdir)
    g = cuda_binding.Generator(0)
    try:
        g.set_option(*option)
        g.load_plan(plan, seed)
        if option[0] == "batch_pairs":
            assert g.emitted > 4 * 256
        check_range(g)
    finally:
        g.close()


@pytest.mark.parametrize("rl,qmode", [pytest.param(rl, q, id="rl%d-nch%d-qp%d" % (rl, fast_nch(rl), q)) for rl in EDGE for q in QMODES])
def test_read_length_edges(rl, qmode, built, workdir):
    """Every (NCH, QP) instance of the array mode, forced with fast_qmode, at read lengths on both sides of every 32-cycle chunk
    boundary (the zeroed tail of a slot starts at 32 * NCH)."""
    import torch
    from simuscop_b200 import cuda_binding
    from test_gpu_kernel_matrix import build_case
    scn = build_case("rl%d" % rl, workdir)
    plan = planfile.read_plan(helpers.plan_dumps(scn, "km")[0])
    g = cuda_binding.Generator(0)
    try:
        g.set_option("fast_qmode", qmode)
        g.load_plan(plan, scn["seed"])
        a = check_range(g)
        st = g.stats()
        assert a["reads"].shape[-1] == (rl + 96 + 15) // 16 * 16
        if torch.cuda.get_device_properties(0).shared_memory_per_block_optin == B200_SMEM_OPTIN:
            assert (st["gen_kernel"], st["gen_nch"], st["gen_qmode"]) == (FAST, fast_nch(rl), qmode), st
    finally:
        g.close()


@pytest.mark.parametrize("layout", ["pe", "se"])
@pytest.mark.parametrize("name", ["dense", "big_store", "names", "twin", "pair_ids"])
def test_plan_edges(name, layout, cases):  # noqa: F811
    """Tickets over 1..32 bins with census-emptied bins, positions and fragment counters of 1..10 digits, 64-byte names of every
    byte value, pair IDs past 2^31, 2^32 and 2^33: the pair ranges of test_gpu_plan_edges."""
    from simuscop_b200 import cuda_binding
    case = cases(name, layout)
    g = cuda_binding.Generator(0)
    try:
        load(g, case)
        for lo, hi, _, _ in case["jobs"][:8]:
            check_range(g, lo, hi)
    finally:
        g.close()


@pytest.mark.parametrize("layout", ["pe", "se"])
def test_ranges_and_pair_ids(layout, profiles):  # noqa: F811
    """Arbitrary [lo, hi), including bins the census empties or thins: pair_id holds exactly the planned IDs of the pairs the
    FASTQ range holds (the oracle's trace); an empty range writes nothing; two handles on two shards concatenate to the
    single-handle arrays."""
    import torch
    from simuscop_b200 import cuda_binding
    plan, _ = dense_case(profiles[layout], layout, True)
    _, _, info = oracle(plan, trace=True)
    ids = info["trace"][:, 0].astype(np.int64)
    g = cuda_binding.Generator(0)
    g2 = cuda_binding.Generator(0)
    try:
        g.load_plan(plan, SEED)
        whole = check_range(g)
        assert (whole["pair_id"].cpu().numpy() == ids).all()
        rng = np.random.default_rng(5)
        for lo, hi in [(0, 1), (int(ids[3]), int(ids[3]) + 1)] + [tuple(sorted(rng.integers(0, g.planned + 1, 2))) for _ in range(6)]:
            a = check_range(g, int(lo), int(hi))
            assert (a["pair_id"].cpu().numpy() == ids[(ids >= lo) & (ids < hi)]).all(), (lo, hi)
        # empty ranges: nothing written
        for lo, hi in ((0, 0), (5, 5), (g.planned, g.planned)):
            out = prefilled(g, 4)
            a = g.generate_reads(lo, hi, out=out)
            assert a["reads"].shape[0] == 0
            assert (out["reads"] == 0xFF).all() and (out["pair_id"] == -1).all() and (out["length"] == -1).all()
        # two shards on two handles
        g2.load_plan(plan, SEED)
        mid = int(ids[len(ids) // 2]) + 1
        parts = [g.generate_reads(0, mid), g2.generate_reads(mid, g.planned)]
        for k in ("reads", "length", "pair_id", "segment", "pos", "frag"):
            assert torch.equal(torch.cat([p[k] for p in parts]), whole[k]), k
    finally:
        g.close()
        g2.close()


def test_stream_order(gen, workdir):
    """Work queued on the caller's stream before the call comes first: a long sleep, then a fill of the output with 0xFF on
    stream s, then generate_reads(stream=s) -- the arrays are the generated ones, not the fill."""
    import torch
    plan, seed = scenario_plan("pe_xten", workdir)
    gen.load_plan(plan, seed)
    want = check_range(gen)
    n = want["reads"].shape[0]
    out = gen.empty_reads(n)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)
        for k in ("reads", "length", "pair_id", "segment", "pos", "frag"):
            out[k].fill_(-1 if out[k].dtype.is_signed else 0xFF)
        a = gen.generate_reads(stream=s, out=out)
    torch.cuda.synchronize()
    for k in ("reads", "length", "pair_id", "segment", "pos", "frag"):
        assert torch.equal(a[k], want[k]), k
    # torch's current stream, taken when no stream is given
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)
        out["reads"].fill_(0xFF)
        a = gen.generate_reads(out=out)
    torch.cuda.synchronize()
    assert torch.equal(a["reads"], want["reads"])


def _k4_plan(workdir):
    d = os.path.join(workdir, "arr_k4")
    os.makedirs(d, exist_ok=True)
    ref = os.path.join(d, "ref.fa")
    synth.make_genome(ref, [40000], seed=31)
    prof = os.path.join(d, "synthetic.profile")
    synth.write_profile(prof, seed=4, kmer=4, read_length=100, bins=3, n_live_qual=7)
    kw = dict(ref=ref, profile=prof, layout="PE", coverage=2, insertSize=250, threads=1, verbose=0, name="k4")
    return planfile.read_plan(helpers.plan_dumps(dict(dir=d, kw=kw, seed=5, name="k4"), "k4")[0])


def test_errors_leave_the_handle_usable(built, workdir):
    """Short capacity, wrong pitch, a null or misaligned pointer, no plan, force_generic, fp64_search and a K = 4 profile are
    refused with the right code and a message naming the limit, before anything is written; the handle then still produces
    the right FASTQ and arrays."""
    import torch
    from simuscop_b200 import cuda_binding
    L = cuda_binding.lib()
    scn = helpers.build_scenario("pe_tiny", workdir)
    plans, ref_out = helpers.reference_run(scn, tag="arr")
    plan, seed = planfile.read_plan(plans[0]), scn["seed"]
    r1, r2 = (helpers.read_file(p) for p in helpers.sample_files(ref_out, plan, 0, scn))

    def raw(g, out, pitch=None, **ptrs):
        p = {k: out[k].data_ptr() for k in ("reads", "length", "pair_id", "segment", "pos", "frag")}
        p.update(ptrs)
        st = abi.ReadArrays(p["reads"], p["length"], p["pair_id"], p["segment"], p["pos"], p["frag"], out["reads"].shape[0],
                            out["reads"].shape[-1] if pitch is None else pitch)
        n = C.c_int64(-7)
        rc = L.ssc_generate_reads(g.h, 0, g.planned, C.byref(st), None, C.byref(n))
        return rc, L.ssc_last_error().decode(), n.value

    g = cuda_binding.Generator(0)
    try:
        # no plan
        with pytest.raises(cuda_binding.SscError, match="ssc error 3"):
            g.read_shape()
        g.load_plan(plan, seed)
        n, mates, pitch = g.read_shape()
        out = prefilled(g, n)
        for what, kw, msg in (("pitch", dict(pitch=pitch + 16), "pitch"), ("null", dict(reads=None), "null"),
                              ("misaligned", dict(reads=out["reads"].data_ptr() + 8), "aligned")):
            rc, err, got = raw(g, out, **kw)
            assert rc == 1 and msg in err and got == -7, (what, rc, err)
        short = prefilled(g, n - 1)
        with pytest.raises(cuda_binding.SscError, match="ssc error 1.*capacity"):
            g.generate_reads(out=short)
        torch.cuda.synchronize()
        assert (out["reads"] == 0xFF).all() and (short["reads"] == 0xFF).all()
        g.set_option("force_generic", 1)
        with pytest.raises(cuda_binding.SscError, match="ssc error 1.*force_generic"):
            g.generate_reads()
        g.set_option("force_generic", 0)
        f1, f2 = g.generate()
        assert f1 == r1 and f2 == r2
        check_range(g)
        # a K = 4 profile, then a plan the fast kernel runs on the same handle
        g.load_plan(_k4_plan(workdir), 5)
        with pytest.raises(cuda_binding.SscError, match="ssc error 1.*kmer 4"):
            g.generate_reads()
        g.load_plan(plan, seed)
        check_range(g)
    finally:
        g.close()
    g = cuda_binding.Generator(0)
    try:
        rc, err, got = raw(g, out)                                 # no plan yet
        assert rc == 3 and "ssc_set_plan" in err and got == -7, (rc, err)
        g.set_option("fp64_search", 1)
        g.load_plan(plan, seed)
        with pytest.raises(cuda_binding.SscError, match="ssc error 1.*fp64_search"):
            g.generate_reads()
        f1, f2 = g.generate()                                      # the FP64 kernel's FASTQ (the option holds for the plan)
        assert f1 == r1 and f2 == r2
    finally:
        g.close()


def test_memory_is_bookkeeping_only(profiles):  # noqa: F811
    """A fresh handle, default batch size, an XTen plan of 2 M pairs: generate_reads adds less than 100 MB of device memory beyond
    the caller's arrays (no FASTQ slab, blob scratch or pinned host slab -- those would take gigabytes), and writes the same
    reads as ssc_generate over a slice of the plan."""
    import torch
    from simuscop_b200 import cuda_binding
    from test_gpu_plan_edges import random_genome
    base = profiles["pe"]
    genome = random_genome(20000, seed=3)
    b = Builder(True)
    b.segment(b"@mem#chr1#", huge_bins(2 << 20, True, genome.size))
    plan = b.plan(base, genome)
    g = cuda_binding.Generator(0)
    try:
        g.load_plan(plan, SEED)
        assert g.emitted >= 1 << 20
        out = g.empty_reads(g.emitted)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(0)[0]
        a = g.generate_reads(out=out)
        torch.cuda.synchronize()
        grew = free0 - torch.cuda.mem_get_info(0)[0]
        assert grew < 100 << 20, "generate_reads took %d MB of device memory" % (grew >> 20)
        assert a["reads"].shape[0] == g.emitted and g.stats()["pairs_emitted"] == g.emitted
        f1, f2 = g.generate(0, 4096)
        a1, a2 = to_fastq(g, {k: v[:4096] for k, v in a.items()})
        assert a1 == f1 and a2 == f2
    finally:
        g.close()
