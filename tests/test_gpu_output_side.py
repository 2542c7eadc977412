"""The output side of the fast kernel against the C oracle (oracle/ssc_oracle.c) on hand-built plans, byte for byte, at the edges
of the kernels that turn its per-ticket blobs into files:

a. move_blobs_tma_kernel, the concurrent mover: it pulls a blob in 4 KB pieces through a ring of 3 stages, so blobs of 1..5
   pieces, the second ring round (over 12 288 bytes) and each warp's per-stage parity bits carried across blobs of different
   piece counts; mover widths of 1, 2, 9 (the default) and 64 SMs, and 0 (the stand-alone move_blobs_kernel);
b. scan_blobs_kernel: rounds of 8 192 lengths, with a partial last round;
c. deflate_blobs_kernel: every gzip member equal to the host mirror's (ssc_gzip_member_host, fitted to the same sample), and
   members that the Huffman code would expand (bytes the sample lacks) written as one stored block.

Every case asserts the coverage it claims from the oracle's records.  Blob j of a batch goes to mover warp j % (16 * SMs), and
the mover moves every batch of a call but the last."""
import ctypes as C
import gzip
import os
import re
import zlib

import numpy as np
import pytest

import helpers
from simuscop_b200 import planfile, synth, testdata
from test_gpu_kernel_matrix import FAST, assert_same_fastq
from test_gpu_plan_edges import NO_MOD, Builder, load, oracle, profiles, records, run_case  # noqa: F401 (profiles: fixture)

pytestmark = pytest.mark.gpu

TICKET = 32                    # FG_CHUNK: pairs per ticket, one blob per ticket and file
PIECE = 4096                   # MV_PIECE: bytes per bulk copy of the mover
STAGES = 3                     # MV_STAGES: ring stages per mover warp
MOVER_WARPS = 16               # MV_WARPS: mover warps per SM
DEFAULT_MOVER = 9
SCAN_ROUND = 8192              # lengths per round of scan_blobs_kernel
DEFAULT_BATCH = 1 << 20
STORED_EXTRA = 23              # gzip header + stored block header + trailer
GZ_HEADER = b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff"

SHORT = b"@"
LONG = b"@" + bytes(range(0x41, 0x5b)) + bytes(range(0x61, 0x7b)) + b"0123456789_"        # 64 bytes of ASCII
ABSENT = b"@" + bytes(range(0x80, 0xbf))                                                  # 64 bytes no sample carries
assert len(LONG) == len(ABSENT) == 64


def always_fast(stats, mode, rl):
    assert stats["gen_kernel"] == FAST, stats


def write_base(workdir, tag, layout, profile=None, ins3=None, **kw):
    """A plan of the front end whose profile header and tables the hand-built plans take.  ins3: an insertion rate with every
    insertion 3 bases long, so that reads grow by 3 per event (32 events, the per-read limit, are 96 bases: the other limit)."""
    d = os.path.join(workdir, "output_side_" + tag)
    os.makedirs(d, exist_ok=True)
    ref = os.path.join(d, "ref.fa")
    synth.make_genome(ref, [5000], seed=31)
    if profile:
        prof = os.path.join(testdata.materialize(os.path.join(workdir, "data")), testdata.PROFILES[profile])
    else:
        prof = os.path.join(d, "synthetic.profile")
        if ins3:
            kw.update(ins_rate=ins3, del_rate=0, n_ins=4)
        synth.write_profile(prof, kmer=3, **kw)
        if ins3:
            with open(prof) as f:
                text = re.sub(r"(\[Insert Frequency\]\n)[^\n]*", "\\g<1>0\t0\t0\t1", f.read())
            with open(prof, "w") as f:
                f.write(text)
    args = dict(ref=ref, profile=prof, layout=layout, coverage=1, insertSize=300 if layout == "PE" else 150, threads=1,
                verbose=0, name="p")
    return planfile.read_plan(helpers.plan_dumps(dict(dir=d, kw=args, seed=1, name=tag), "p")[0])


@pytest.fixture(scope="module")
def bases(profiles, workdir):
    out = {"xten": profiles["pe"],
           "gaiix": write_base(workdir, "gaiix", "PE", "GAIIx"),
           "se33": write_base(workdir, "se33", "SE", seed=33, read_length=33, bins=31, n_live_qual=7),
           "k3_160": write_base(workdir, "k3_160", "PE", seed=160, read_length=160, bins=40, n_live_qual=7),
           "k3_160_ins": write_base(workdir, "k3_160_ins", "PE", seed=161, read_length=160, bins=40, n_live_qual=7, ins3=0.105)}
    for k, rl in [("xten", 151), ("gaiix", 74), ("se33", 33), ("k3_160", 160), ("k3_160_ins", 160)]:
        b = out[k]
        assert b.hdr["read_length"] == rl and b.hdr["kmer"] == 3, k
        assert not b.paired or b.hdr["min_insert_size"] >= rl, k          # no bin below is risky: emitted == planned
    return out


def acgt(n, seed):
    return np.frombuffer(b"ACGT", np.uint8)[np.random.default_rng(seed).integers(0, 4, n)].copy()


def build(base, genome, segs, seed):
    """segs: [(name, pairs, (lo, hi))]: a segment of `pairs` pairs in bins of 1..4 pairs that lie in genome[lo:hi]."""
    RL = base.hdr["read_length"]
    mx = base.hdr["min_insert_size"] + base.hdr["n_isize"] - 1 if base.paired else 0
    b = Builder(base.paired)
    names = {}
    rng = np.random.default_rng(seed)
    for name, pairs, (lo, hi) in segs:
        if name not in names:
            names[name] = b.name(name)
        bins = []
        while pairs > 0:
            k = min(pairs, int(rng.integers(1, 5)))
            w = int(rng.integers(RL, 400))
            sp = int(rng.integers(lo, hi - mx - RL - w))
            bins.append((0, genome.size, sp, sp + w, NO_MOD, k))
            pairs -= k
        b.segment(names[name], bins)
    return b.plan(base, genome)


def make_case(plan):
    """The oracle's files and the byte offset of every record (pair) in them."""
    o1, o2, info = oracle(plan)
    P = plan.planned_pairs()
    assert info["emitted"] == P
    if b"\n" in plan.names:          # names with line feeds: the records of the oracle pair by pair
        lens = np.array([[len(x) for x in oracle(plan, i, i + 1)[:2]] for i in range(P)])
        rec = tuple(np.concatenate(([0], np.cumsum(lens[:, f]))) for f in range(2))
    else:
        rec = (records(o1), records(o2))
    assert rec[0][-1] == len(o1) and rec[1][-1] == len(o2) and len(rec[0]) == P + 1
    return dict(plan=plan, chunk=None, emitted=P, o=(o1, o2), rec=rec if plan.paired else (rec[0], None))


def slab_pairs(case, batch_pairs):
    n = min(batch_pairs, max(case["emitted"], 1))
    return -(-n // TICKET) * TICKET


def batches(case, lo, hi, batch_pairs):
    B = slab_pairs(case, batch_pairs)
    return [(e, min(hi, e + B)) for e in range(lo, hi, B)]


def blob_lens(case, lo, hi):
    """[(file 1 length, file 2 length)] of the tickets of the batch [lo, hi)."""
    out = []
    for t in range(lo, hi, TICKET):
        e = min(hi, t + TICKET)
        out.append(tuple(int(r[e] - r[t]) if r is not None else 0 for r in case["rec"]))
    return out


def pieces(n):
    return -(-n // PIECE)


def moved_batches(case, calls, batch_pairs):
    """[[(file 1 length, file 2 length) per ticket] of every batch the mover moves]: every batch of a call but the last."""
    return [blob_lens(case, blo, bhi) for lo, hi in calls for blo, bhi in batches(case, lo, hi, batch_pairs)[:-1]]


def mover_work(case, calls, batch_pairs, ctas):
    """warp -> [piece count of every blob it moves, in order] over the calls."""
    W = MOVER_WARPS * ctas
    work = {}
    for lens in moved_batches(case, calls, batch_pairs):
        for j, ls in enumerate(lens):
            work.setdefault(j % W, []).extend(pieces(n) for n in ls if n)
    return work


def expected(case, lo, hi):
    o, r = case["o"], case["rec"]
    return tuple(o[f][r[f][lo]:r[f][hi]] if r[f] is not None else b"" for f in range(2))


def run_plain(case, calls, options, what):
    """Every call against the oracle through ssc_generate, then through ssc_generate_device: byte counts, and the mover's
    kernel time.  Returns the statistics of the device calls."""
    from simuscop_b200 import cuda_binding
    g = cuda_binding.Generator(0)
    try:
        for k, v in options.items():
            g.set_option(k, v)
        load(g, case)
        for lo, hi in calls:
            got, want = g.generate(lo, hi), expected(case, lo, hi)
            if got != want:            # (first_diff walks the bytes in Python: only to report a difference)
                assert_same_fastq(got, want, "%s, pairs [%d, %d), %s" % (what, lo, hi, options))
        g.reset_stats()
        for lo, hi in calls:
            want = expected(case, lo, hi)
            d = g.generate_device(lo, hi)
            assert (d["bytes1"], d["bytes2"]) == tuple(len(x) for x in want), d
        st = g.stats()
        always_fast(st, "fast", case["plan"].hdr["read_length"])
        return st
    finally:
        g.close()


# ---------------------------------------------------------------------------------------------------------------------------
# a. the mover: piece counts 1..5, the second ring round, parity carried across blobs of different piece counts
# ---------------------------------------------------------------------------------------------------------------------------
# profile -> piece counts of the blobs it moves: short names and 64-byte names in alternating segments
PIECE_CASES = {"se33": {1, 2}, "xten": {3, 4}, "k3_160": {3, 4}, "k3_160_ins": {4, 5}}
assert set().union(*PIECE_CASES.values()) == {1, 2, 3, 4, 5}


@pytest.fixture(scope="module")
def piece_cases(bases):
    cache = {}

    def get(name):
        if name not in cache:
            base = bases[name]
            n = 300000
            genome = acgt(n, 3)
            if name == "k3_160_ins":       # 64-byte names only: reads of 160 + ~3 x 17 bases, blobs of 15.6..16.4 KB
                segs = [(LONG, int(x), (0, n)) for x in np.random.default_rng(4).integers(20, 300, 12)]
            else:
                segs = [([SHORT, LONG][i % 2], int(x), (0, n)) for i, x in enumerate(np.random.default_rng(4).integers(20, 700, 24))]
            case = make_case(build(base, genome, segs, 5))
            if name == "k3_160_ins":
                RL = base.hdr["read_length"]
                longest = max(len(s) for o in case["o"] for s in o.split(b"\n")[1::4])
                assert longest == RL + 96, longest       # at the per-read limits (32 events of 3 bases): the slab holds them
            cache[name] = case
        return cache[name]
    return get


@pytest.mark.parametrize("name", PIECE_CASES)
def test_mover_piece_counts(name, piece_cases):
    """Blobs of 1..5 pieces on the mover (one SM: 16 warps, each moving many blobs in turn), the whole plan and a call that
    starts and ends inside a ticket; some warp moves a 4- or 5-piece blob (a second ring round) right after a blob of another
    piece count, and the reverse."""
    case = piece_cases(name)
    P = case["emitted"]
    calls = [(0, P), (TICKET * 7 + 5, P - 19)]
    batch = TICKET * MOVER_WARPS * 2 + 13
    work = mover_work(case, calls, batch, 1)
    moved = set().union(*work.values())
    assert PIECE_CASES[name] <= moved, (name, sorted(moved))
    if max(PIECE_CASES[name]) >= 4:
        pairs = [(a, b) for seq in work.values() for a, b in zip(seq, seq[1:])]
        assert any(b >= 4 and a != b for a, b in pairs), name
        assert any(a >= 4 and a != b for a, b in pairs), name
    st = run_plain(case, calls, {"concurrent_move": 1, "batch_pairs": batch}, "pieces %s" % name)
    assert st["mover_kernel_ms"] > 0, st


# ---------------------------------------------------------------------------------------------------------------------------
# mover widths: one blob per warp and batch, at least four, a batch size that is not a multiple of 32, a call inside tickets
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def width_case(bases):
    n = 400000
    segs = [([SHORT, LONG][i % 2], int(x), (0, n)) for i, x in enumerate(np.random.default_rng(6).integers(100, 3000, 190))]
    case = make_case(build(bases["xten"], acgt(n, 7), segs, 8))
    assert case["emitted"] > 2 * (4 * MOVER_WARPS * 64 + 1) * TICKET
    return case


@pytest.mark.parametrize("per_warp", ["one", "four"])
@pytest.mark.parametrize("ctas", [0, 1, 2, DEFAULT_MOVER, 64])
def test_mover_widths(ctas, per_warp, width_case):
    """concurrent_move 1, 2, 9 (the default) and 64 SMs, and 0 (the stand-alone move after every batch), with batches of as
    many tickets as the mover has warps (one blob per warp) or of 4 per warp + 1 (13 pairs past a multiple of 32)."""
    case = width_case
    W = MOVER_WARPS * max(ctas, 1)
    batch = TICKET * W if per_warp == "one" else TICKET * 4 * W + 13
    P = case["emitted"]
    calls = [(0, P), (TICKET * 101 + 17, P - TICKET * 3 - 9)]
    moved = moved_batches(case, calls, batch)
    assert len(moved) >= 2 * len(calls) - 1 and len(moved) >= 2
    tickets = [len(b) for b in moved]                  # tickets of a moved batch: blob j goes to warp j % W
    if per_warp == "one":
        assert set(tickets) == {W}, tickets
    else:
        assert set(tickets) == {4 * W + 1}, tickets
    st = run_plain(case, calls, {"concurrent_move": ctas, "batch_pairs": batch}, "width %d %s" % (ctas, per_warp))
    assert (st["mover_kernel_ms"] > 0) == (ctas > 0), st


# ---------------------------------------------------------------------------------------------------------------------------
# b. scan rounds
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def scan_case(bases):
    n = 200000
    P = 16385 * TICKET + 777
    return make_case(build(bases["se33"], acgt(n, 9), [(SHORT, P // 4, (0, n)), (LONG, P // 4, (0, n)),
                                                       (SHORT, P - 2 * (P // 4), (0, n))], 10))


@pytest.mark.parametrize("tickets", [SCAN_ROUND - 1, SCAN_ROUND, SCAN_ROUND + 1, 2 * SCAN_ROUND + 1])
def test_scan_rounds(tickets, scan_case):
    """Batches of 8191, 8192, 8193 and 16385 tickets: one round, one full round, a round of one length, two rounds + one; the
    last batch of the call is partial too."""
    P = scan_case["emitted"]
    assert P > tickets * TICKET and P % (tickets * TICKET)
    case = dict(scan_case, jobs=[(0, P) + expected(scan_case, 0, P)])
    run_case(case, "fast", {"batch_pairs": tickets * TICKET}, always_fast, "scan %d" % tickets, device_bytes=True)


# ---------------------------------------------------------------------------------------------------------------------------
# c. gzip members
# ---------------------------------------------------------------------------------------------------------------------------
def split_members(z):
    out = []
    while z:
        d = zlib.decompressobj(wbits=31)
        d.decompress(z)
        assert d.eof
        n = len(z) - len(d.unused_data)
        out.append(z[:n])
        z = z[n:]
    return out


def host_member(blob, sample):
    buf = C.create_string_buffer(len(blob) + 4096)
    from simuscop_b200 import cuda_binding
    m = cuda_binding.lib().ssc_gzip_member_host(blob, len(blob), sample, len(sample), buf, len(buf))
    assert m > 0
    return buf.raw[:m]


def run_gzip(case, calls, batch_pairs, what):
    """Every call in gzip mode: inflates to the oracle's bytes, and every member equals the host mirror's, built with the
    sample the library fits its table to.  Returns [(raw blob, member)]."""
    from simuscop_b200 import cuda_binding
    o, r = case["o"], case["rec"]
    files = 2 if case["plan"].paired else 1
    B = slab_pairs(case, batch_pairs if batch_pairs else DEFAULT_BATCH)
    lo0 = calls[0][0]
    first = min(calls[0][1], lo0 + B)
    s_hi = min(first, lo0 + 256 * TICKET)
    sample = b"".join(o[f][r[f][lo0]:r[f][s_hi]] for f in range(files))
    out = []
    g = cuda_binding.Generator(0)
    try:
        g.set_option("gzip", 1)
        if batch_pairs:
            g.set_option("batch_pairs", batch_pairs)
        load(g, case)
        for lo, hi in calls:
            z = g.generate(lo, hi)
            want = expected(case, lo, hi)
            got = tuple(gzip.decompress(x) for x in z)
            if got != want:
                assert_same_fastq(got, want, "%s, pairs [%d, %d)" % (what, lo, hi))
            tickets = [(t, min(bhi, t + TICKET)) for blo, bhi in batches(case, lo, hi, B) for t in range(blo, bhi, TICKET)]
            for f in range(files):
                members = split_members(z[f])
                blobs = [o[f][r[f][t]:r[f][e]] for t, e in tickets]
                assert len(members) == len(blobs), (len(members), len(blobs))
                for j, (blob, m) in enumerate(zip(blobs, members)):
                    assert m == host_member(blob, sample), "%s, call [%d, %d), file %d, member %d of %d bytes (blob %d)" % (
                        what, lo, hi, f + 1, j, len(m), len(blob))
                    assert len(m) <= len(blob) + STORED_EXTRA
                    out.append((blob, m))
        always_fast(g.stats(), "fast", case["plan"].hdr["read_length"])
    finally:
        g.close()
    return out


@pytest.fixture(scope="module")
def gzip_cases(bases, piece_cases, profiles):
    from test_gpu_plan_edges import names_case
    cache = {}

    def get(name):
        if name not in cache:
            if name == "names":
                cache[name] = make_case(names_case(profiles["pe"]))
            elif name in ("xten", "k3_160"):
                cache[name] = piece_cases(name)
            else:
                n = 200000
                segs = [([SHORT, LONG][i % 2], int(x), (0, n)) for i, x in enumerate(np.random.default_rng(12).integers(20, 500, 16))]
                cache[name] = make_case(build(bases[name], acgt(n, 13), segs, 14))
        return cache[name]
    return get


GZIP_CASES = {"xten": ("xten", None, False), "xten_batch32": ("xten", 32, False), "xten_batch4096": ("xten", 4096, False),
              "xten_mid_plan": ("xten", None, True), "gaiix": ("gaiix", None, False), "se33": ("se33", None, False),
              "k3_160_names64": ("k3_160", None, False), "names": ("names", None, False)}


@pytest.mark.parametrize("name", GZIP_CASES)
def test_gzip_members_equal_host_mirror(name, gzip_cases):
    """deflate_blobs_kernel's members equal ssc_gzip_member_host's byte for byte (table fitted to both files of the first
    min(tickets, 256) tickets of the first batch of the first call): XTen <5,8>, GAIIx <3,16>, SE, RL 160 with 64-byte names,
    names of every byte value, batches of one ticket, of 4096 pairs and the default, and a first call that starts mid-plan;
    blob lengths of every residue mod 8 (the kernel codes the tail bytes 0-3 and 4-7 apart)."""
    key, batch, mid = GZIP_CASES[name]
    case = gzip_cases(key)
    P = case["emitted"]
    calls = [(P // 3 + 5, P - 11), (0, P // 3 + 5)] if mid else [(0, P)]
    got = run_gzip(case, calls, batch, name)
    if len(got) >= 256:
        assert {len(b) % 8 for b, _ in got} == set(range(8))


# ---------------------------------------------------------------------------------------------------------------------------
# members that coding would expand
# ---------------------------------------------------------------------------------------------------------------------------
EXPANDING_BATCH = 64 * TICKET


@pytest.fixture(scope="module")
def expanding_cases(bases):
    """256 tickets of ACGT reads with short names (the sample holds no other bytes, whatever the batch size), then 64 tickets
    of reads in an N run whose 64-byte names carry bytes absent from the sample."""
    cache = {}

    def get(name):
        if name not in cache:
            n, nrun = 200000, 60000
            genome = acgt(n + nrun, 15)
            genome[n:] = ord("N")
            plan = build(bases[name], genome, [(b"@normal#chr1#", 256 * TICKET, (0, n)), (ABSENT, 64 * TICKET, (n, n + nrun))], 16)
            case = make_case(plan)
            sample = b"".join(o[:r[256 * TICKET]] for o, r in zip(case["o"], case["rec"]))
            assert not set(ABSENT[1:]) & set(sample) and b"N" not in b"".join(sample.split(b"\n")[1::4])
            cache[name] = case
        return cache[name]
    return get


@pytest.mark.parametrize("batch", ["one_ticket", "default", "only_expanding"])
@pytest.mark.parametrize("name", ["xten", "k3_160"])
def test_gzip_expanding_members_are_stored(name, batch, expanding_cases):
    """Tickets whose Huffman code (14-15 bits for every byte the sample lacks) would be longer than the blob: each member is
    one stored block of raw + 23 bytes, equal to the host mirror's, and the file inflates to the oracle's bytes; in batches of
    one ticket, of the default size and of 64 tickets (the fifth batch holds nothing but such tickets)."""
    case = expanding_cases(name)
    bp = {"one_ticket": TICKET, "default": None, "only_expanding": EXPANDING_BATCH}[batch]
    got = run_gzip(case, [(0, case["emitted"])], bp, "expanding %s %s" % (name, batch))
    stored = [(b, m) for b, m in got if (m[10] >> 1) & 3 == 0]
    assert stored and all(m[:11] == GZ_HEADER + b"\x01" and len(m) == len(b) + STORED_EXTRA for b, m in stored)
    assert any(ABSENT in b for b, _ in stored) and not any(ABSENT in b for b, m in got if (m[10] >> 1) & 3 == 2)
