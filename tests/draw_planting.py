"""Profiles whose thresholds sit exactly on the draws the reads make (shared by test_draw_thresholds and
test_gpu_draw_thresholds).

Every random choice of a read compares a 32-bit Philox word u with thresholds T that the host derives from the FP64 CDFs
(symbol = #{i : T[i] < u}), or is the FP64 fragment position.  Whether a device form of that compare uses < or <=, or keeps
the + 1 of a limit, only shows when u == T, which a random draw meets with probability 2^-32.  Since
r(u) = ZERO_FINAL + (1 - ZERO_FINAL) * u / 2^32 (the reference's randomDouble) is strictly increasing in u, a CDF entry of r(u)
compresses to the threshold T = u exactly; and since Philox is a pure function of (seed, pair, mate, stream, index) and the
oracle's draw trace says which table row every draw reads, the tables can be built so that chosen draws land on their
thresholds: "at" (T = u, the draw takes the lower symbol) or "one past" (T = u - 1, the higher one).

The builder plants in the order in which the decisions depend on one another (insert size -> indel lengths -> substitution
rows -> quality rows), running the traced oracle between the steps.  Each planted threshold is recorded as a Planted entry, so
that the tests can count how many draws of the final plan sit on one, and move each by one."""
import os
from collections import namedtuple

import numpy as np

import helpers
from simuscop_b200 import planfile, synth

ZERO_FINAL = 2.2204e-16
TWO32 = 4294967296.0
MASK = 0xFFFFFFFF
STREAM_FRAG, STREAM_CYCLE, STREAM_LEN = 0, 1, 2
SEED = 11

# site: "isize", "inslen", "dellen", "sub", "qual"; row: the table row the draw reads (see row_keys); slot: index of the
# threshold in the row's compressed CDF; kind: "at" (T = u), "past" (T = u - 1), and for 16-bit keys "key_below"
# (T = (u & 0xFFFF0000) - 1: the key alone says u > T), "key_above" (T = (u | 0xFFFF) + 1: the key alone says u < T), "key_tie"
# (T = u | 0xFFFF: the key ties, the exact repeat decides u <= T)
Planted = namedtuple("Planted", "site row slot T u kind")


# ---------------------------------------------------------------------------------------------------------------------------
# Philox4x32-10, vectorised (the oracle's ssco_block address layout)
# ---------------------------------------------------------------------------------------------------------------------------
def philox(c0, c1, c2, c3, k0, k1):
    c0, c1, c2, c3 = (np.asarray(x, dtype=np.uint64) & MASK for x in np.broadcast_arrays(c0, c1, c2, c3))
    k0, k1 = np.uint64(k0 & MASK), np.uint64(k1 & MASK)
    m0, m1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    s32, mk = np.uint64(32), np.uint64(MASK)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2
        c0, c1, c2, c3 = (p1 >> s32) ^ c1 ^ k0, p1 & mk, (p0 >> s32) ^ c3 ^ k1, p0 & mk
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & mk, (k1 + np.uint64(0xBB67AE85)) & mk
    return [x.astype(np.uint32) for x in (c0, c1, c2, c3)]


def block(seed, pair, mate, stream, blk, index):
    pair = np.asarray(pair, dtype=np.uint64)
    c2 = (np.asarray(mate, dtype=np.uint64) << np.uint64(28)) | np.uint64(stream << 24) | np.asarray(blk, dtype=np.uint64)
    return philox(pair & np.uint64(MASK), pair >> np.uint64(32), c2, index, seed & MASK, seed >> 32)


# ---------------------------------------------------------------------------------------------------------------------------
# CDF rows that compress to chosen thresholds
# ---------------------------------------------------------------------------------------------------------------------------
def r(u):
    """The reference's draw of u on [ZERO_FINAL, 1) (no FMA: numpy rounds each operation)."""
    return ZERO_FINAL + (1.0 - ZERO_FINAL) * (np.float64(u) / TWO32)


def cdf_row(T, syms, n):
    """A CDF of n entries whose compressed form is thresholds T (ascending, < 2^32 - 1) for syms[:-1], then syms[-1] for the
    rest: entries below syms[0] are 0, entry syms[-1] and above are 1."""
    assert len(syms) == len(T) + 1 and list(syms) == sorted(set(syms)) and syms[-1] < n
    assert all(a < b for a, b in zip(T, T[1:])) and T[-1] < MASK if len(T) else True
    c = np.zeros(n)
    for i, s in enumerate(syms):
        c[s:] = r(T[i]) if i < len(T) else 1.0
    return c


def threshold_of(u, kind):
    return {"at": u, "past": u - 1, "key_below": (u & 0xFFFF0000) - 1, "key_above": (u | 0xFFFF) + 1,
            "key_tie": u | 0xFFFF}[kind]


def choose(draws, n, rng, kinds, slot_phase=0):
    """n distinct draws spread over the sorted draws of a row (every slot of the row gets one) and their thresholds:
    [(slot, T, u, kind)] with kinds[(slot + slot_phase) % len(kinds)]; None when the row cannot take n strictly ascending
    thresholds."""
    d = np.unique(np.asarray(draws, dtype=np.int64))
    d = d[(d > 0) & (d < MASK - 0x10000)]
    if d.size < n:
        return None
    idx = np.sort(rng.choice(d.size, size=n, replace=False))
    out = []
    for slot, u in enumerate(d[idx]):
        kind = kinds[(slot + slot_phase) % len(kinds)]
        out.append((slot, threshold_of(int(u), kind), int(u), kind))
    Ts = [t for _, t, _, _ in out]
    if not all(a + 1 < b for a, b in zip(Ts, Ts[1:])) or Ts[0] < 1:     # room for a move by one either way
        return None
    return out


# ---------------------------------------------------------------------------------------------------------------------------
# plans
# ---------------------------------------------------------------------------------------------------------------------------
# name -> synthetic profile, layout, genome and coverage; live: quality symbols per planted row
PROFILES = {
    "pe151": dict(kw=dict(kmer=3, read_length=151, bins=45, n_live_qual=8, bases="ACTG"), layout="PE", live=8,
                  lengths=(30000, 6000), coverage=8),
    "pe64": dict(kw=dict(kmer=3, read_length=64, bins=31, n_live_qual=40, bases="GATC"), layout="PE", live=40,
                 lengths=(60000, 9000), coverage=14),
    "se97": dict(kw=dict(kmer=3, read_length=97, bins=49, n_live_qual=6, bases="TGCA"), layout="SE", live=6,
                 lengths=(40000, 8000), coverage=8),
    "k5": dict(kw=dict(kmer=5, read_length=100, bins=3, n_live_qual=7, bases="ACGT"), layout="PE", live=7,
               lengths=(40000, 6000), coverage=6),
}
RATE_PROFILES = ("pe151", "pe64")


def base_plan(name, workdir, small=False):
    """A plan of the C++ front end on the synthetic profile of PROFILES[name] (`small`: a short genome for the rate cases)."""
    spec = PROFILES[name]
    d = os.path.join(workdir, "dt_%s%s" % (name, "_small" if small else ""))
    os.makedirs(d, exist_ok=True)
    ref = os.path.join(d, "ref.fa")
    lengths = [6000, 2000] if small else list(spec["lengths"])
    synth.make_genome(ref, lengths, seed=43, n_runs=1, lower_runs=1, run_len=150, iupac=10)
    prof = os.path.join(d, "synthetic.profile")
    synth.write_profile(prof, seed=sum(map(ord, name)), ins_rate=3e-3, del_rate=3e-3, **spec["kw"])
    rl = spec["kw"]["read_length"]
    kw = dict(ref=ref, profile=prof, layout=spec["layout"], coverage=4 if small else spec["coverage"], insertSize=rl + 90,
              threads=1, verbose=0, name="dt")
    return planfile.read_plan(helpers.plan_dumps(dict(dir=d, kw=kw, seed=5, name=name), "dt")[0])


def with_tables(plan, **changes):
    """A copy of `plan` (sharing bins, segments, names and genome) with header fields and tables replaced."""
    p = planfile.Plan()
    p.hdr, p.tables = dict(plan.hdr), dict(plan.tables)
    for k, v in changes.items():
        if k in p.tables:
            p.tables[k] = np.ascontiguousarray(v, dtype=np.float64)
        else:
            p.hdr[k] = v
    p.genome, p.bins, p.segs, p.names = plan.genome, plan.bins, plan.segs, plan.names
    return p


def oracle(plan, trace=True):
    from oracle import binding as oracle_binding
    return oracle_binding.generate(plan, SEED, draw_trace=trace)


def row_keys(site, info, plan):
    """(row keys, draws) of every decision of `site` in a traced oracle run."""
    if site == "isize":
        f = info["frag"]
        return np.zeros(len(f), dtype=np.int64), f["x1"]
    if site in ("inslen", "dellen"):
        s = info["scan"]
        s = s[s["kind"] == (1 if site == "inslen" else 2)]
        return np.zeros(len(s), dtype=np.int64), s["lenword"]
    b = info["base"]
    B = plan.hdr["bins"]
    if site == "sub":
        b = b[b["row"] >= 0]
        return ((b["subtab"] - 1) * plan.hdr["n_kmer_rows"] + b["row"]) * B + b["bin"], b["u2"]
    b = b[b["qrow"] >= 0]
    return b["qrow"] * B + b["bin"], b["u3"]


def group(keys, draws):
    order = np.argsort(keys, kind="stable")
    k, d = keys[order], draws[order]
    cut = np.flatnonzero(np.diff(k)) + 1
    return {int(kk[0]): dd for kk, dd in zip(np.split(k, cut), np.split(d, cut)) if kk.size}


KINDS = ("at", "past")
KEY_KINDS = ("at", "key_below", "past", "key_tie", "at", "key_above", "past")


def plant_case(name, workdir):
    """(plan, [Planted]) for PROFILES[name]: insert sizes (PE), insertion and deletion lengths, substitution rows and quality
    rows planted on the draws of the reads."""
    spec = PROFILES[name]
    plan = base_plan(name, workdir)
    RL = plan.hdr["read_length"]
    rng = np.random.default_rng(sum(map(ord, name)) + 1)
    planted = []

    # 1. insert sizes: 39 thresholds on attempt-0 x1 words of distinct pairs.  The table starts 2 below the read length,
    # so that threshold 1 separates a rejected attempt (fragment of RL - 1) from an accepted one: the census's decision too
    if plan.paired:
        _, _, info = oracle(plan)
        f = info["frag"]
        f = f[f["attempt"] == 0]
        ch = choose(f["x1"], 39, rng, KINDS)
        T = [t for _, t, _, _ in ch]
        plan = with_tables(plan, n_isize=40, min_insert_size=RL - 2, isize_cdf=cdf_row(T, list(range(40)), 40))
        planted += [Planted("isize", 0, s, t, u, k) for s, t, u, k in ch]

    # 2. insertion / deletion lengths, on the length words of the first event of each read (its position does not depend on
    # any length): 11 and 19 thresholds, every symbol live
    _, _, info = oracle(plan)
    s = info["scan"]
    ev = s[s["kind"] > 0]
    _, first = np.unique(ev["pair"] * 2 + ev["mate"], return_index=True)
    ev = ev[first]
    changes = {}
    for site, kind, n, tab in (("inslen", 1, plan.hdr["n_ins"], "ins_cdf"), ("dellen", 2, plan.hdr["n_del"], "del_cdf")):
        ch = choose(ev["lenword"][ev["kind"] == kind], n - 1, rng, KINDS, slot_phase=kind)
        T = [t for _, t, _, _ in ch]
        changes[tab] = cdf_row(T, list(range(n)), n)
        planted += [Planted(site, 0, sl, t, u, k) for sl, t, u, k in ch]
    plan = with_tables(plan, **changes)

    # 3. substitution rows: three thresholds on draws of the row, or (every fifth row) a leading 0 and two, so base > 0
    _, _, info = oracle(plan)
    keys, draws = row_keys("sub", info, plan)
    B, R = plan.hdr["bins"], plan.hdr["n_kmer_rows"]
    tabs = {1: plan.tables["subs_cdf1"].reshape(-1, 4).copy()}
    if plan.hdr["use_cdf2"]:
        tabs[2] = plan.tables["subs_cdf2"].reshape(-1, 4).copy()
    for i, (key, d) in enumerate(sorted(group(keys, draws).items())):
        lead = i % 5 == 4
        ch = choose(d, 2 if lead else 3, rng, KINDS, slot_phase=i)
        if ch is None:
            continue
        T = [t for _, t, _, _ in ch]
        tab, row = divmod(key, R * B)
        tabs[tab + 1][row] = cdf_row(T, [1, 2, 3] if lead else [0, 1, 2, 3], 4)
        planted += [Planted("sub", key, sl + (1 if lead else 0), t, u, k) for sl, t, u, k in ch]
    plan = with_tables(plan, subs_cdf1=tabs[1].ravel(), **({"subs_cdf2": tabs[2].ravel()} if 2 in tabs else {}))

    # 4. quality rows: `live` symbols, every threshold slot planted; rows of more than 8 symbols (the 16-bit-key tables) also
    # take thresholds decided by the keys alone and key ties
    _, _, info = oracle(plan)
    keys, draws = row_keys("qual", info, plan)
    live, Q = spec["live"], plan.hdr["n_qual"]
    qt = plan.tables["quality_cdf"].reshape(-1, Q).copy()
    kinds = KEY_KINDS if live > 8 else KINDS
    for i, (key, d) in enumerate(sorted(group(keys, draws).items())):
        ch = choose(d, live - 1, rng, kinds, slot_phase=i)
        if ch is None:
            continue
        lo = int(rng.integers(0, Q - live))
        syms = sorted(rng.choice(np.arange(lo, min(Q, lo + 2 * live)), size=live, replace=False).tolist())
        qt[key] = cdf_row([t for _, t, _, _ in ch], syms, Q)
        planted += [Planted("qual", key, sl, t, u, k) for sl, t, u, k in ch]
    plan = with_tables(plan, quality_cdf=qt.ravel())
    return plan, planted


def coverage(plan, planted, info):
    """{(site, kind): planted thresholds whose draw the final plan makes in the planted row} and the same per (site, slot,
    kind)."""
    seen = {}
    for site in {p.site for p in planted}:
        keys, draws = row_keys(site, info, plan)
        seen[site] = set(zip(keys.tolist(), draws.tolist()))
    total, per_slot = {}, {}
    for p in planted:
        if (p.row, p.u) in seen[p.site]:
            total[(p.site, p.kind)] = total.get((p.site, p.kind), 0) + 1
            per_slot[(p.site, p.slot, p.kind)] = per_slot.get((p.site, p.slot, p.kind), 0) + 1
    return total, per_slot


def move_by_one(plan, planted, site):
    """The plan with every "at" / "past" threshold of `site` moved by one (at -> past, past -> at): what an off-by-one
    compare of that site on the device amounts to."""
    tables = {"isize": "isize_cdf", "inslen": "ins_cdf", "dellen": "del_cdf"}
    sel = [p for p in planted if p.site == site and p.kind in KINDS]
    if site in tables:
        c = plan.tables[tables[site]].copy()
        for p in sel:
            c[c == r(p.T)] = r(p.T - 1 if p.kind == "at" else p.T + 1)
        return with_tables(plan, **{tables[site]: c})
    B, R = plan.hdr["bins"], plan.hdr["n_kmer_rows"]
    if site == "sub":
        tabs = {1: plan.tables["subs_cdf1"].reshape(-1, 4).copy()}
        if plan.hdr["use_cdf2"]:
            tabs[2] = plan.tables["subs_cdf2"].reshape(-1, 4).copy()
        for p in sel:
            tab, row = divmod(p.row, R * B)
            c = tabs[tab + 1][row]
            c[c == r(p.T)] = r(p.T - 1 if p.kind == "at" else p.T + 1)
        return with_tables(plan, subs_cdf1=tabs[1].ravel(), **({"subs_cdf2": tabs[2].ravel()} if 2 in tabs else {}))
    Q = plan.hdr["n_qual"]
    qt = plan.tables["quality_cdf"].reshape(-1, Q).copy()
    for p in sel:
        c = qt[p.row]
        c[c == r(p.T)] = r(p.T - 1 if p.kind == "at" else p.T + 1)
    return with_tables(plan, quality_cdf=qt.ravel())


def records(data):
    lines = data.split(b"\n")
    return [b"\n".join(lines[i:i + 4]) for i in range(0, len(lines) - 1, 4)]


def differing_records(a, b):
    n = 0
    for x, y in zip(a, b):
        ra, rb = records(x), records(y)
        assert len(ra) == len(rb)
        n += sum(p != q for p, q in zip(ra, rb))
    return n


# ---------------------------------------------------------------------------------------------------------------------------
# rate cases: the same bins, only the rates and the length tables differ
# ---------------------------------------------------------------------------------------------------------------------------
def _scan(plan):
    return oracle(plan)[2]["scan"]


def _lenword(scan_row, which):
    w = block(SEED, int(scan_row["pair"]), int(scan_row["mate"]), STREAM_LEN, 0, int(scan_row["j"]))
    return int(w[which])


def _one_past_table(word, n=2):
    """A length table that gives `word` length 1 (threshold word - 1) and length 0 to every draw below it."""
    return cdf_row([word - 1], [0, 1], n) if word > 0 else cdf_row([], [1], n)


def _quotient_in(del_rate, ir, lo, hi):
    q = np.float64(del_rate) / (np.float64(1.0) - np.float64(ir))
    return lo < q <= hi


def _del_rate_for(ir, lo, hi):
    """A del_rate whose FP64 quotient del_rate / (1 - insert_rate) lies in (lo, hi]."""
    x = np.float64(hi) * (np.float64(1.0) - np.float64(ir))
    for _ in range(64):
        if _quotient_in(x, ir, lo, hi):
            return float(x)
        q = x / (1.0 - ir)
        x = np.nextafter(x, -np.inf) if q > hi else np.nextafter(x, np.inf)
    raise AssertionError("no del_rate for (%r, %r]" % (lo, hi))


def rate_cases(name, workdir):
    """name -> (plan, expected events: ("ins" / "del", pair, mate, j) or None for "no event at all", or "edge").
    The thresholds of the insertion and deletion tests sit on u*, the smallest x0 (or x1) any scanned position draws."""
    base = base_plan(name, workdir, small=True)
    RL = base.hdr["read_length"]
    zero = with_tables(base, insert_rate=0.0, del_rate=0.0, n_ins=2, ins_cdf=[0.0, 1.0], n_del=2, del_cdf=[0.0, 1.0])
    s = _scan(zero)
    assert (s["kind"] == 0).all() or (s["x0"][s["kind"] == 1] == 0).all()
    i = int(np.argmin(s["x0"]))
    ustar = int(s["x0"][i])
    cases = {}
    cases["ins_at"] = (with_tables(zero, insert_rate=ustar / TWO32, ins_cdf=_one_past_table(_lenword(s[i], 0))),
                       ("ins",) + tuple(int(s[i][k]) for k in ("pair", "mate", "j")))
    cases["ins_below"] = (with_tables(zero, insert_rate=(ustar - 1) / TWO32), None)
    for tag, ir in (("", 0.0), ("_ir", (ustar - 1) / TWO32)):
        tested = s[s["x0"] / TWO32 > ir]                        # positions whose deletion test runs
        k = int(np.argmin(tested["x1"]))
        v = int(tested["x1"][k])
        at = _del_rate_for(ir, v / TWO32, (v + 1) / TWO32)
        below = _del_rate_for(ir, (v - 1) / TWO32, v / TWO32)
        cases["del_at" + tag] = (with_tables(zero, insert_rate=ir, del_rate=at, del_cdf=_one_past_table(_lenword(tested[k], 1))),
                                 ("del",) + tuple(int(tested[k][c]) for c in ("pair", "mate", "j")))
        cases["del_below" + tag] = (with_tables(zero, insert_rate=ir, del_rate=below), None)
    # limit edges: a test that passes everywhere (the limit 2^32 wraps: every read takes the slow path) and the largest limit
    # that does not wrap.  Length tables mostly 0, with thresholds planted on the top length words (at and one past)
    lw = np.sort([_lenword(row, 0) for row in s[:4000]])[-12:]
    ins_T = [int(lw[j]) - (i & 1) for i, j in enumerate((0, 5, 10))]
    ins_cdf = cdf_row(ins_T, [0, 1, 2, 5], 6)
    cases["ins_wrap"] = (with_tables(zero, insert_rate=1.0, n_ins=6, ins_cdf=ins_cdf), "edge")
    cases["ins_max"] = (with_tables(zero, insert_rate=(TWO32 - 2) / TWO32, n_ins=6, ins_cdf=ins_cdf), "edge")
    # the deletion test everywhere (del_rate 1, insert_rate 0: delT = 2^32 - 1): lengths of 3, RL - 49 (the read falls below
    # 50 bases: every event of it is undone) and RL + 4 (clipped at the read end), planted on the words of read starts
    dw = np.sort([_lenword(row, 1) for row in s[s["j"] == 0][:600]])[-9:]
    del_T = [int(dw[j]) - (i & 1) for i, j in enumerate((0, 4, 8))]
    n_del = RL + 5
    cases["del_wrap"] = (with_tables(zero, del_rate=1.0, n_del=n_del, del_cdf=cdf_row(del_T, [0, 3, RL - 49, RL + 4], n_del)),
                         "edge")
    return cases


# ---------------------------------------------------------------------------------------------------------------------------
# position cases: the FP64 position spos + span * u / 2^32 is one more than the exact quotient's floor
# ---------------------------------------------------------------------------------------------------------------------------
POS_STORE = (1 << 25) + (1 << 13)
POS_PAIRS = 12000        # pair IDs searched for every kind
POS_DOUBLE_PAIRS = 160000  # pair IDs searched for the rare double rounding


def fp64_pos(spos, span, u):
    return int(np.float64(spos) + np.float64(span) * (np.float64(u) / TWO32))


def exact_pos(spos, span, u):
    return (spos * (1 << 32) + span * u) >> 32


def fma_pos(spos, span, u):
    """The position as one fused multiply-add would give it: spos + span * u / 2^32 rounded once (int / int division rounds
    correctly)."""
    return int((spos * (1 << 32) + span * u) / (1 << 32))


# kind -> (span range, spos for draw u): "product": the product rounds up to an integer; "sum": the sum does; "double": the
# product rounds to exactly half a unit of the sum, which rounds up to the even integer, while the exact sum (a fused
# multiply-add) is just below that half and rounds down
POSITION_KINDS = {
    "double": (((1 << 21), (1 << 22)), lambda u: (1 << 24) + (u % ((1 << 24) - (1 << 22) - 1000))),
    "product": (((1 << 22), (1 << 25)), lambda u: 1000 + (u % 5000)),
    "sum": ((2, (1 << 21)), lambda u: (1 << 24) + (u % ((1 << 24) - (1 << 21) - 1000))),
}


def position_solution(u, kinds=tuple(POSITION_KINDS)):
    """(kind, spos, span) for which the FP64 position of draw u is one more than the exact floor (for "double": and the fused
    form is not), from span * u = -n (mod 2^32) for small n; None if there is none."""
    tz = (u & -u).bit_length() - 1
    inv = pow(u >> tz, -1, 1 << 32)
    for kind in kinds:
        (lo, hi), spos_of = POSITION_KINDS[kind]
        spos = spos_of(u)
        for n in range(1, 17 if kind == "double" else 40):
            if n % (1 << tz):
                continue
            span = ((-(n >> tz)) * inv) % (1 << (32 - tz))
            while span < hi:
                if span >= lo and spos + span + 600 < POS_STORE:
                    exact = exact_pos(spos, span, u)
                    if fp64_pos(spos, span, u) == exact + 1 and (kind != "double" or fma_pos(spos, span, u) == exact):
                        return kind, spos, span
                span += 1 << (32 - tz)
    return None


def position_case(base, rng_seed=3):
    """A hand-built PE plan of one-pair bins on a random store of 2^25 + 2^13 bases: the pair IDs whose attempt-0 draw has a
    rounding solution (any kind among the first POS_PAIRS, the double rounding up to POS_DOUBLE_PAIRS) get a bin with that spos and span (every third one with the contig end where the exact position would
    leave RL bases and the FP64 one leaves RL - 1: the census rejects attempt 0); the other pair IDs sit in bins whose contig
    is shorter than a read (the census empties them).  Returns (plan, [(pair, spos, span, u, kind, end_case)])."""
    from test_gpu_plan_edges import Builder, NO_MOD, random_genome
    RL = base.hdr["read_length"]
    genome = random_genome(POS_STORE, seed=rng_seed)
    genome = np.where((genome >= ord("a")) & (genome <= ord("z")), genome - 32, genome).astype(np.uint8)
    ids = np.arange(POS_DOUBLE_PAIRS, dtype=np.uint64)
    x0 = block(SEED, ids, 0, STREAM_FRAG, 0, 0)[0]
    b = Builder(True)
    nm = b.name(b"@pos#chr1#")
    dead = (POS_STORE - RL // 2, POS_STORE)            # a contig shorter than a read
    pending, cases = 0, []
    for pid in range(POS_DOUBLE_PAIRS):
        u = int(x0[pid])
        if pid >= POS_PAIRS and not (u >> 31 and u & 1):
            pending += 1
            continue
        sol = position_solution(u, tuple(POSITION_KINDS) if pid < POS_PAIRS else ("double",))
        if sol is None:
            pending += 1
            continue
        kind, spos, span = sol
        if pending:
            b.segment(nm, [(dead[0], dead[1], 0, 3, NO_MOD, pending)])
            pending = 0
        epos = spos + span - 1
        end_case = len(cases) % 3 == 2
        exact = exact_pos(spos, span, u)
        ce = exact + RL if end_case else POS_STORE - RL
        b.segment(nm, [(0, ce, spos, epos, NO_MOD, 1)])
        cases.append((pid, spos, span, u, kind, end_case))
    if pending:
        b.segment(nm, [(dead[0], dead[1], 0, 3, NO_MOD, pending)])
    plan = b.plan(base, genome)
    return plan, cases
