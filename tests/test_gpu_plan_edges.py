"""The generation kernels against the C oracle (oracle/ssc_oracle.c) on hand-built plans, byte for byte, where the plan rather
than the profile drives the hot path outside what the front end produces on a realistic job:

a. dense bins: bins of one pair next to bins of 31..65 pairs, so that the 32 pairs of a ticket of the fast kernel span every
   number of bins from 1 to 32 (the shuffle search of the ticket prologue runs all five of its steps), bins that plan no pair,
   bins the census empties (every attempt fails: their pair IDs are used up, nothing is emitted) or thins (attempts > 0),
   segments of 1, 2, 31, 32 and 33 bins, pair ranges that start and end at every offset of a ticket, batches of one ticket;
b. read-name fields: positions at the digit boundaries 10^k - 1 / 10^k up to 2^31 - 1 on a store of 2^31 + 4 Mbases, the
   modulus of the position (segsize) below it, fragment counters at the digit boundaries up to 0x7fffffff, names of 1..64 bytes
   carrying every byte value but NUL, a 64-byte name that ends on the last byte of a 131 071-byte name blob; in gzip mode too;
c. pair IDs (the Philox counter) past 2^31, 2^32 and 2^33.

Every case runs on the fast kernel with and without the concurrent blob mover, on the generic kernel and on the FP64 search,
and asserts through ssc_stats which of them ran.  The oracle walks every pair of a segment it emits from, so the plans put
their large pair counts in segments the oracle steps over: huge leading segments for (c), and for the fragment counters of
(b) a twin plan in which the leading bins of a segment form a segment of their own (same name, same pair IDs, same draws): the
counters of the twin's tail segment are those of the real plan minus the pairs of the leading bins.

The plans obey two rules of ssc_set_plan: a bin is "risky" (its pairs go through the census) when a fragment drawn from it can
end past its contig, when an SE bin is narrower than a read, or when the insert sizes reach below the read length; and the
census total stays below 2^31.  So every bin with a huge count is non-risky: the XTen profile's insert-size table starts at
the read length, and the SE bins are at least a read wide."""
import ctypes as C
import gzip
import os

import numpy as np
import pytest

import helpers
from simuscop_b200 import abi, planfile, synth, testdata
from test_gpu_kernel_matrix import B200_SMEM_OPTIN, FAST, FP64, GENERIC_SMEM, assert_same_fastq, fast_nch

pytestmark = pytest.mark.gpu

SEED = 11
TICKET = 32                   # FG_CHUNK: pairs per ticket of the fast kernel
GEN_TILE_PAIRS = 32           # the smallest batch_pairs
NAME_BLOB_LIMIT = (1 << 17) - 1
I32 = 0x7fffffff
NO_MOD = 0xFFFFFFFF           # a segsize above every position: pos % segsize is pos
MAX_INSERT = 451              # XTen: insert sizes 151..451 (table of 301 entries from the read length)
CHUNK = 4 << 20               # the large store repeats one 4 MiB chunk

MODES = {"fast": {}, "no_mover": {"concurrent_move": 0}, "generic": {"force_generic": 1}, "fp64": {"fp64_search": 1}}
GZIP_MODE = {"gzip": {"gzip": 1}}


def random_genome(n, seed, runs=4):
    """ACGT with runs of N and of lower case."""
    rng = np.random.default_rng(seed)
    g = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].copy()
    for _ in range(runs):
        a = int(rng.integers(0, max(1, n - 300)))
        g[a:a + int(rng.integers(20, 300))] = ord("N")
        a = int(rng.integers(0, max(1, n - 3000)))
        g[a:a + int(rng.integers(100, 3000))] += 32
    return g


@pytest.fixture(scope="module")
def profiles(built, workdir):
    """layout -> a plan of the front end whose profile header and tables the hand-built plans take: XTen RL 151 PE (runs
    generate_slots_kernel<5,8>) and a synthetic K = 3 SE profile with RL 64."""
    out = {}
    for layout in ("pe", "se"):
        d = os.path.join(workdir, "pe_profile_" + layout)
        os.makedirs(d, exist_ok=True)
        ref = os.path.join(d, "ref.fa")
        synth.make_genome(ref, [5000], seed=31)
        if layout == "pe":
            prof = os.path.join(testdata.materialize(os.path.join(workdir, "data")), testdata.PROFILES["XTen"])
        else:
            prof = os.path.join(d, "synthetic.profile")
            synth.write_profile(prof, seed=64, kmer=3, read_length=64, bins=31, n_live_qual=7)
        kw = dict(ref=ref, profile=prof, layout=layout.upper(), coverage=1, insertSize=300 if layout == "pe" else 150,
                  threads=1, verbose=0, name="p")
        out[layout] = planfile.read_plan(helpers.plan_dumps(dict(dir=d, kw=kw, seed=1, name=layout), "p")[0])
    assert out["pe"].hdr["min_insert_size"] >= out["pe"].hdr["read_length"] == 151 and out["pe"].hdr["n_isize"] > 0
    assert out["pe"].hdr["min_insert_size"] + out["pe"].hdr["n_isize"] - 1 <= MAX_INSERT
    assert out["se"].hdr["read_length"] == 64 and not out["se"].paired
    return out


class Builder:
    """Bins, segments and the name blob of a plan, segment by segment."""

    def __init__(self, paired):
        self.paired = paired
        self.bins, self.segs, self.names = [], [], bytearray()

    def name(self, nm):
        off = len(self.names)
        self.names += nm
        return off, len(nm)

    def segment(self, name, bins):
        """name: bytes, or (offset, length) of a name already in the blob; bins: (hap_base, contig_end, spos, epos, segsize,
        pairs) with pairs <= 0 for a read_count of that value."""
        off, ln = self.name(name) if isinstance(name, (bytes, bytearray)) else name
        s = len(self.segs)
        self.segs.append((len(self.bins), len(bins), off, ln))
        for hb, ce, sp, ep, ss, n in bins:
            self.bins.append((hb, ce, sp, ep, ss, self.read_count(n), s, 0))
        return s

    def read_count(self, pairs):
        # PE: 2n and 2n - 1 reads both make n pairs; never 2^31 - 1 reads, whose pair count (n + 1) / 2 overflows the
        # oracle's int
        if pairs <= 0 or not self.paired:
            return pairs
        return 2 * pairs - (pairs & 1 if pairs < (1 << 30) - 1 else 0)

    def plan(self, base, genome):
        p = planfile.Plan()
        p.hdr, p.tables = base.hdr, base.tables
        p.genome = genome
        p.bins = np.array(self.bins, dtype=abi.BIN_DTYPE)
        p.segs = np.array(self.segs, dtype=abi.SEG_DTYPE)
        p.names = bytes(self.names)
        return p


def max_pairs(paired):
    return (1 << 30) - 1 if paired else I32


def huge_bins(pairs, paired, contig):
    """Non-risky bins that plan `pairs` pairs in all, each as large as a bin can be."""
    out, m = [], max_pairs(paired)
    while pairs > 0:
        n = min(pairs, m)
        out.append((0, contig, 1000, 5000, NO_MOD, n))
        pairs -= n
    return out


def pair_bases(plan):
    rc = np.maximum(plan.bins["read_count"].astype(np.int64), 0)
    per = (rc + 1) // 2 if plan.paired else rc
    return np.concatenate(([0], np.cumsum(per)))


def records(data):
    """Byte offset of every record of a FASTQ file (names without line feeds), and the end."""
    nl = np.flatnonzero(np.frombuffer(data, np.uint8) == 10)
    return np.concatenate(([0], nl[3::4] + 1))


def header_fields(data):
    """(position field, fragment counter) of every record header of a file whose names are ASCII without line feeds."""
    out = []
    for h in data.split(b"\n")[0::4][:-1]:
        _, pos, frag = h.rsplit(b"#", 2)
        out.append((pos, frag.split(b"/")[0]))
    return out


def shift_counters(data, by):
    """The same records with every fragment counter increased by `by` (parsed from the right of the header)."""
    lines = data.split(b"\n")
    for i in range(0, len(lines) - 1, 4):
        head, _, tail = lines[i].rpartition(b"#")
        num, slash, mate = tail.partition(b"/")
        lines[i] = head + b"#" + str(int(num) + by).encode() + slash + mate
    return b"\n".join(lines)


# ---------------------------------------------------------------------------------------------------------------------------
# a. dense bins
# ---------------------------------------------------------------------------------------------------------------------------
def dense_case(base, layout, with_census):
    """A few thousand bins, most of one pair; the bins of 31..65 pairs are placed so that each starts at every offset of a
    ticket (emitted-pair index mod 32) once per size.  with_census adds bins with read_count 0 and negative, bins the census
    empties (their contig is shorter than a read) and bins next to a contig end that fail some attempts."""
    paired = base.paired
    RL = base.hdr["read_length"]
    rng = np.random.default_rng(5 if paired else 6)
    main, short, tail = 200000, RL - 10, 8000             # contigs: a long one, one shorter than a read, one for near-end bins
    genome = random_genome(main + short + tail, seed=17)
    c_short, c_tail = (main, main + short), (main + short, main + short + tail)
    frag = MAX_INSERT if paired else 0

    def ordinary(n):
        w = int(rng.integers(RL, 1000)) if not paired else int(rng.integers(0, 1000))
        sp = int(rng.integers(0, main - frag - RL - w))
        return (0, main, sp, sp + w, 0, n)

    def special():
        """(bin, pairs it emits): a few failures per bin never reach the census's limit of 1000"""
        kind = int(rng.integers(0, 4))
        if kind == 0:
            return (0, main, 10, 2000, 0, int(rng.choice([0, -1, -7]))), 0
        if kind == 1:
            return (c_short[0], c_short[1], 0, 5, 0, int(rng.integers(1, 4))), 0
        hb, ce = c_tail
        sp = tail - (300 if paired else RL + 60)
        n = int(rng.integers(1, 5))
        return (hb, ce, sp, sp + (200 if paired else RL + 30), 0, n), n

    specs, emitted = [], 0
    for size in [31, 32, 33, 63, 64, 65]:
        for off in rng.permutation(TICKET):
            singles = TICKET * int(rng.integers(1, 3))
            while (emitted - int(off)) % TICKET or singles > 0:
                specs.append(ordinary(1))
                emitted += 1
                singles -= 1
                if with_census and rng.random() < 0.05:
                    spec, n = special()
                    specs.append(spec)
                    emitted += n
            specs.append(ordinary(size))
            emitted += size
    specs += [ordinary(1) for _ in range(3 * TICKET)]        # a ticket of 32 bins
    seg_sizes = [1, 2, 31, 32, 33, 7, 100]
    b = Builder(paired)
    i = s = 0
    while i < len(specs):
        k = seg_sizes[s % len(seg_sizes)]
        segsize = [main, 1000, 7, 1, NO_MOD, 999999][s % 6]
        b.segment(b"@dense%d#chr%d#" % (s, s % 3), [x[:4] + (segsize,) + x[5:] for x in specs[i:i + k]])
        i += k
        s += 1
    return b.plan(base, genome), s


def ticket_bin_counts(plan, pair_ids):
    """Distinct bins in each ticket of 32 emitted pairs of the whole plan."""
    bins = np.searchsorted(pair_bases(plan), pair_ids, side="right") - 1
    return [len(np.unique(bins[j:j + TICKET])) for j in range(0, len(bins), TICKET)]


def dense_ranges(pair_ids):
    """(e_lo, e_hi) emitted-index ranges: the start at every offset of a ticket, the end at every offset too."""
    out = []
    n = len(pair_ids)
    for j in range(TICKET):
        lo = (TICKET * 13 * j) % (n - 400) // TICKET * TICKET + j
        end_off = (7 * j + 3) % TICKET
        hi = lo + 1 + (end_off - lo - 1) % TICKET + TICKET * (j % 5)
        out.append((lo, hi))
    return out


# ---------------------------------------------------------------------------------------------------------------------------
# b / c. read-name fields and pair IDs
# ---------------------------------------------------------------------------------------------------------------------------
def digit_positions():
    return sorted({p for k in range(1, 10) for p in (10 ** k - 1, 10 ** k)} | {I32})


def big_store_case(base, chunk, reps):
    """Positions at the digit boundaries up to 2^31 - 1 on a store of `reps` copies of `chunk`, and positions above the modulus
    of the read name (segsize 1, 7, 10^9, and one that leaves exactly 10^9).  One segment per bin."""
    paired = base.paired
    RL = base.hdr["read_length"]
    total = chunk.size * reps
    b = Builder(paired)
    nm = b.name(b"@big#chr9#")
    mods = [(I32, 1), (I32, 7), (I32, 10 ** 9), (I32, I32 - 10 ** 9), (I32, I32), (I32, I32 + 1), (10 ** 9, 10 ** 9 - 1),
            (10 ** 9 - 1, 10 ** 9)]
    for p, segsize in [(p, NO_MOD) for p in digit_positions()] + mods:
        if paired:
            b.segment(nm, [(0, total, p, p, segsize, 3)])        # one start position, three draws of the insert size
        else:
            # SE: a fragment is the bin, so the bin is a read wide and straddles the boundary
            sp = max(0, min(p - 40, I32 - 80))
            b.segment(nm, [(0, total, sp, sp + 80, segsize, 12)])
    assert max(x[3] for x in b.bins) + MAX_INSERT + RL < total
    return b.plan(base, None)


def names_case(base):
    """Names of 1, 2, 31, 32, 33, 63 and 64 bytes that carry every byte value 0x01..0xFF after the '@', in a blob of exactly
    131 071 bytes whose last segment's 64-byte name ends on its last byte."""
    paired = base.paired
    RL = base.hdr["read_length"]
    n = 60000
    genome = random_genome(n, seed=23)
    b = Builder(paired)
    rng = np.random.default_rng(8)
    byte = 0
    lengths = [1, 2, 31, 32, 33, 63, 64] * 2
    names = []
    for L in lengths:
        nm = bytearray(b"@")
        for _ in range(L - 1):
            nm.append(byte % 255 + 1)
            byte += 1
        names.append(bytes(nm))
    last = b"@" + bytes(range(0xC1, 0x100))
    assert len(last) == 64

    def bins():
        out = []
        for _ in range(3):
            w = int(rng.integers(RL, 600))
            sp = int(rng.integers(0, n - MAX_INSERT - RL - w))
            out.append((0, n, sp, sp + w, int(rng.integers(500, 70000)), int(rng.integers(1, 5))))
        return out
    for nm in names:
        b.segment(nm, bins())
    b.names += bytes(NAME_BLOB_LIMIT - 64 - len(b.names))
    b.segment(last, bins())
    assert len(b.names) == NAME_BLOB_LIMIT and b.segs[-1][2] + 64 == NAME_BLOB_LIMIT
    assert set(b"".join(names + [last])) == set(range(1, 256))
    return b.plan(base, genome)


def twin_case(base, extra=0):
    """(plan A, plan B, [(tail segment of B, pairs of the leading bins)]): in A a segment is leading bins L followed by tail
    bins T; in B, L and T are two segments with the same name and segsize.  The counters of T run over 10^k - 1 / 10^k for
    k = 1..9, and the last one ends at exactly 0x7fffffff (plus `extra`)."""
    paired = base.paired
    RL = base.hdr["read_length"]
    n = 40000
    genome = random_genome(n, seed=29)
    rng = np.random.default_rng(9)
    tails = [(10 ** k - 4, 8) for k in range(1, 10)] + [(I32 - 8, 8 + extra)]
    A, B = Builder(paired), Builder(paired)
    meta = []
    for i, (lead, nt) in enumerate(tails):
        name = b"@twin%d#chr%d#" % (i, i)
        segsize = [NO_MOD, 9973][i % 2]
        lead_bins = [x[:4] + (segsize, x[5]) for x in huge_bins(lead, paired, n)]
        tail_bins = []
        left = nt
        while left > 0:
            k = min(left, 3)
            sp = int(rng.integers(0, n - MAX_INSERT - RL - 400))
            tail_bins.append((0, n, sp, sp + int(rng.integers(RL, 400)), segsize, k))
            left -= k
        A.segment(name, lead_bins + tail_bins)
        nmB = B.name(name)
        B.segment(nmB, lead_bins)
        meta.append((B.segment(nmB, tail_bins), lead))
    return A.plan(base, genome), B.plan(base, genome), meta


PAIR_ID_EDGES = [[1 << 31], [(1 << 32) - 1, 1 << 32], [(1 << 33) + 5]]


def pair_id_case(base):
    """Huge leading segments (which the oracle steps over), then a small segment around each group of PAIR_ID_EDGES."""
    paired = base.paired
    RL = base.hdr["read_length"]
    n = 40000
    genome = random_genome(n, seed=37)
    rng = np.random.default_rng(10)
    b = Builder(paired)
    planned = 0
    for g, edges in enumerate(PAIR_ID_EDGES):
        lead = edges[0] - 37 - planned
        while lead > 0:
            k = min(lead, I32)
            b.segment(b"@lead#chr%d#" % g, huge_bins(k, paired, n))
            lead -= k
        small = []
        for _ in range(40):
            sp = int(rng.integers(0, n - MAX_INSERT - RL - 300))
            small.append((0, n, sp, sp + int(rng.integers(RL, 300)), 7919, int(rng.integers(1, 4))))
        b.segment(b"@ids%d#chr%d#" % (g, g), small)
        planned = int(pair_bases(b.plan(base, genome))[-1])
        assert planned > edges[-1] + 20
    return b.plan(base, genome)


# ---------------------------------------------------------------------------------------------------------------------------
# expected bytes: each case is (how to load it, planned / emitted pairs, [(pair_lo, pair_hi, FASTQ 1, FASTQ 2)])
# ---------------------------------------------------------------------------------------------------------------------------
def periodic_window(chunk, lo, hi):
    return chunk[np.arange(lo, hi, dtype=np.int64) % chunk.size]


def oracle(plan, lo=0, hi=None, genome=None, first=0, trace=False):
    """The oracle over the upper-cased store (or window): the reference upper-cases every haplotype string, while the device
    packs either case, so the device gets the lower-case runs as they are."""
    from oracle import binding as oracle_binding
    g = plan.genome if genome is None else genome
    g = np.where((g >= ord("a")) & (g <= ord("z")), g - 32, g).astype(np.uint8)
    return oracle_binding.generate(plan, SEED, lo, hi, trace=trace, genome=g, genome_first=first)


@pytest.fixture(scope="module")
def cases(profiles):
    cache = {}

    def get(name, layout):
        key = (name, layout)
        if key in cache:
            return cache[key]
        base = profiles[layout]
        case = dict(chunk=None, jobs=[])
        if name in ("dense", "dense_plain"):
            plan, nsegs = dense_case(base, layout, name == "dense")
            o1, o2, info = oracle(plan, trace=True)
            ids = info["trace"][:, 0]
            counts = ticket_bin_counts(plan, ids)
            assert max(counts) == TICKET and set(range(1, TICKET + 1)) <= set(counts), sorted(set(counts))
            if name == "dense":
                bases = pair_bases(plan)
                per = np.diff(bases)
                emitted = np.bincount(np.searchsorted(bases, ids, side="right") - 1, minlength=len(per))
                assert ((per > 0) & (emitted == 0)).any(), "no bin emptied by the census"
                assert (info["trace"][:, 1] > 0).any(), "no attempt > 0"
                assert (plan.bins["read_count"] == 0).any() and (plan.bins["read_count"] < 0).any()
            case["jobs"].append((0, plan.planned_pairs(), o1, o2))
            r1, r2 = records(o1), records(o2) if plan.paired else None
            for lo, hi in dense_ranges(ids):
                case["jobs"].append((int(ids[lo]), int(ids[hi - 1]) + 1, o1[r1[lo]:r1[hi]],
                                     o2[r2[lo]:r2[hi]] if plan.paired else b""))
            case["emitted"] = len(ids)
        elif name == "big_store":
            chunk = random_genome(CHUNK, seed=41, runs=40)
            reps = (1 << 31) // CHUNK + 1
            plan = big_store_case(base, chunk, reps)
            case.update(chunk=chunk, reps=reps)
            out1, out2 = [], []
            bases = pair_bases(plan)
            for s in range(len(plan.segs)):
                b = plan.bins[s]
                lo, hi = int(b["spos"]), min(int(b["epos"]) + MAX_INSERT + 1, chunk.size * reps)
                f1, f2, info = oracle(plan, int(bases[s]), int(bases[s + 1]), genome=periodic_window(chunk, lo, hi), first=lo)
                assert info["emitted"] == bases[s + 1] - bases[s]
                out1.append(f1)
                out2.append(f2)
            o1, o2 = b"".join(out1), b"".join(out2)
            digits = {len(p) for p, _ in header_fields(o1)}
            assert digits == set(range(1, 11)), digits
            case["jobs"].append((0, plan.planned_pairs(), o1, o2))
        elif name == "names":
            plan = names_case(base)
            o1, o2, info = oracle(plan)
            case["jobs"].append((0, plan.planned_pairs(), o1, o2))
        elif name == "twin":
            plan, planB, meta = twin_case(base)
            bases = pair_bases(planB)
            segB = planB.segs
            fr = set()
            for s, lead in meta:
                lo = int(bases[segB["first_bin"][s]])
                hi = int(bases[segB["first_bin"][s] + segB["n_bins"][s]])
                f1, f2, info = oracle(planB, lo, hi)
                assert info["emitted"] == hi - lo
                f1, f2 = shift_counters(f1, lead), shift_counters(f2, lead) if plan.paired else b""
                fr |= {int(c) for _, c in header_fields(f1)}
                case["jobs"].append((lo, hi, f1, f2))
            assert {k for k in range(1, 10) if {10 ** k - 1, 10 ** k} <= fr} == set(range(1, 10)) and max(fr) == I32
        elif name == "pair_ids":
            plan = pair_id_case(base)
            ids = []
            for edges in PAIR_ID_EDGES:
                for e in edges:
                    f1, f2, info = oracle(plan, e - 20, e + 20, trace=True)
                    assert info["emitted"] == 40
                    ids += list(info["trace"][:, 0])
                    case["jobs"].append((e - 20, e + 20, f1, f2))
            assert max(ids) >= (1 << 33) and min(ids) < (1 << 31)
        case["plan"] = plan
        case.setdefault("emitted", plan.planned_pairs())
        cache[key] = case
        return case
    return get


def load(g, case):
    """Profile, haplotype store and plan of `case` into Generator g: plan.genome, or `reps` copies of `chunk` built on the
    device (ssc_reference_upload + ssc_genome_append_ref)."""
    from simuscop_b200 import cuda_binding
    plan = case["plan"]
    if case["chunk"] is None:
        g.load_plan(plan, SEED)
        return
    L, ck = cuda_binding.lib(), cuda_binding._ck
    prof = plan.profile_struct()
    ck(L.ssc_set_profile(g.h, C.byref(prof)))
    chunk, reps = case["chunk"], case["reps"]
    ck(L.ssc_genome_reserve(g.h, chunk.size * reps))
    ck(L.ssc_reference_upload(g.h, chunk.tobytes(), chunk.size))
    first = C.c_uint64()
    ck(L.ssc_genome_append_ref(g.h, 0, chunk.size, reps, C.byref(first)))
    assert first.value == 0 and g.genome_size() == chunk.size * reps
    g.set_plan(plan.bins, plan.segs, plan.names, SEED)


@pytest.fixture(scope="module")
def expect_kernel(built):
    """Asserts the kernel a run launched; the instance of the fast kernel where the B200's shared-memory budget holds."""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin

    def check(stats, mode, rl):
        if mode == "generic":
            assert stats["gen_kernel"] == GENERIC_SMEM, stats
        elif mode == "fp64":
            assert stats["gen_kernel"] == FP64, stats
        else:
            assert (stats["gen_kernel"], stats["gen_nch"]) == (FAST, fast_nch(rl)), stats
            if optin == B200_SMEM_OPTIN:
                assert stats["gen_qmode"] == 8, stats
    return check


def run_case(case, mode, options, expect_kernel, what, device_bytes=False):
    from simuscop_b200 import cuda_binding
    plan = case["plan"]
    g = cuda_binding.Generator(0)
    try:
        for k, v in options.items():
            g.set_option(k, v)
        load(g, case)
        assert (g.planned, g.emitted) == (plan.planned_pairs(), case["emitted"])
        for lo, hi, o1, o2 in case["jobs"]:
            f1, f2 = g.generate(lo, hi)
            if options.get("gzip"):
                f1, f2 = gzip.decompress(f1), gzip.decompress(f2)
            assert_same_fastq((f1, f2), (o1, o2), "%s, pairs [%d, %d), %s" % (what, lo, hi, options))
            if device_bytes:
                d = g.generate_device(lo, hi)
                assert (d["bytes1"], d["bytes2"]) == (len(o1), len(o2)), d
        expect_kernel(g.stats(), mode, plan.hdr["read_length"])
    finally:
        g.close()


VARIANTS = {"ranges": {}, "batch_min": {"batch_pairs": GEN_TILE_PAIRS}, "batch_odd": {"batch_pairs": GEN_TILE_PAIRS + 13},
            "one_cta": {"max_ctas": 1}}


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("layout", ["pe", "se"])
def test_dense_bins(layout, mode, variant, cases, expect_kernel):
    """Tickets that span 1..32 bins, with bins of no pair, emptied and thinned by the census, and segments of 1..100 bins:
    the whole plan and 32 pair ranges that start and end at every offset of a ticket, in batches of the default size, of one
    ticket (batch_pairs 32) and of a size that is not a multiple of 32 (rounded up to whole tiles), and on one CTA; the byte
    counts of ssc_generate_device match."""
    case = cases("dense", layout)
    if variant != "ranges":
        case = dict(case, jobs=case["jobs"][:1])
    run_case(case, mode, dict(MODES[mode], **VARIANTS[variant]), expect_kernel, "dense %s %s" % (layout, variant),
             device_bytes=variant == "ranges")


@pytest.mark.parametrize("layout", ["pe", "se"])
def test_dense_bins_without_census(layout, cases, expect_kernel):
    """The dense bins alone (no bin the census handles): every ticket's bin search runs over device bins of full pairs."""
    run_case(cases("dense_plain", layout), "fast", {}, expect_kernel, "dense_plain %s" % layout)


@pytest.mark.parametrize("mode", list(MODES) + list(GZIP_MODE))
@pytest.mark.parametrize("layout", ["pe", "se"])
@pytest.mark.parametrize("name", ["big_store", "names", "twin", "pair_ids"])
def test_plan_fields(name, layout, mode, cases, expect_kernel):
    """big_store: positions of 1..10 digits up to 2^31 - 1 and the modulus below them; names: 1..64 bytes with every byte
    value, a name ending on the last byte of the largest blob; twin: fragment counters of 1..10 digits up to 0x7fffffff;
    pair_ids: pair IDs across 2^31, 2^32 - 1, 2^32 and 2^33 + 5 inside a ticket.  gzip output inflates to the same bytes."""
    run_case(cases(name, layout), mode, dict(MODES, **GZIP_MODE)[mode], expect_kernel, "%s %s" % (name, layout))


def set_plan_error(plan):
    from simuscop_b200 import cuda_binding
    g = cuda_binding.Generator(0)
    try:
        g.load_plan(plan, SEED)
    except cuda_binding.SscError as e:
        return str(e)
    finally:
        g.close()
    return None


def test_plan_rejections(profiles):
    """ssc_set_plan refuses, with SSC_ERR_INVALID, a fragment counter past 0x7fffffff, a name blob of 2^17 bytes, a name of 65
    bytes, of 0 bytes, or one that does not start with '@'; ssc_genome_reserve refuses a store the fast kernel cannot address
    (2^36 bases)."""
    from simuscop_b200 import cuda_binding
    base = profiles["pe"]
    plan, _, _ = twin_case(base)
    assert set_plan_error(plan) is None
    plan, _, _ = twin_case(base, extra=1)
    assert "fragment counter overflow" in set_plan_error(plan)

    def names_plan(blob, off, ln):
        b = Builder(True)
        b.names = bytearray(blob)
        b.segment((off, ln), [(0, 5000, 100, 200, NO_MOD, 2)])
        return b.plan(base, random_genome(5000, seed=3))
    ok = b"@" + b"n" * 63
    assert set_plan_error(names_plan(ok + bytes(NAME_BLOB_LIMIT - 64), 0, 64)) is None
    for blob, off, ln, why in [(ok + bytes(NAME_BLOB_LIMIT + 1 - 64), 0, 64, "name blob of 131072 bytes"),
                               (ok + b"#", 0, 65, "bad name"), (ok, 0, 0, "bad name"), (b"x" + ok, 0, 64, "bad name"),
                               (ok, 1, 63, "bad name")]:
        err = set_plan_error(names_plan(blob, off, ln))
        assert err is not None and "ssc error 1" in err and why in err, (len(blob), off, ln, err)
    g = cuda_binding.Generator(0)
    try:
        prof = base.profile_struct()
        cuda_binding._ck(cuda_binding.lib().ssc_set_profile(g.h, C.byref(prof)))
        with pytest.raises(cuda_binding.SscError, match="ssc error 1: haplotype store"):
            cuda_binding._ck(cuda_binding.lib().ssc_genome_reserve(g.h, 1 << 36))
    finally:
        g.close()
